"""ORACLE - TEST INFRASTRUCTURE ONLY.  Seeded synthetic heat-map / tag-map pairs for the fast_utils checks
(planted persons with per-person tags, optional plateaus and clutter peaks)."""
import numpy as np

JOINT_ORDER_17 = [i - 1 for i in [1, 2, 3, 4, 5, 6, 7, 12, 13, 8, 9, 10, 11, 14, 15, 16, 17]]


def make_case(seed, n=2, c=17, h=48, w=40, people=4, presence=0.85, tagnoise=0.05, spread=2.0, plateau=False,
              clutter=0):
    rs = np.random.RandomState(seed)
    det = (rs.rand(n, c, h, w) * 0.05).astype(np.float32)
    tm = (rs.randn(n, c, h, w) * 0.05).astype(np.float32)
    for i in range(n):
        for p in range(people):
            for j in range(c):
                if rs.rand() > presence:
                    continue
                y, x = rs.randint(2, h - 2), rs.randint(2, w - 2)
                a = np.float32(0.3 + 0.7 * rs.rand())
                det[i, j, y, x] = a
                if plateau and rs.rand() < 0.3:
                    det[i, j, y, x + 1] = a
                tm[i, j, y - 1:y + 2, x - 1:x + 2] = np.float32(p * spread + rs.randn() * tagnoise)
        for _ in range(clutter):
            j = rs.randint(c)
            y, x = rs.randint(0, h), rs.randint(0, w)
            det[i, j, y, x] = np.float32(0.1 + 0.4 * rs.rand())
    return det, tm


def joint_order(c):
    return [j for j in JOINT_ORDER_17 if j < c][:c]


# (seed, kwargs, threshold, window, max_count, tag_threshold) - every case keeps counts and persons <= 10 so that the
# reference's own arrays are not overrun
GOLDEN_CASES = [
    (1, dict(people=1), 0.1, 5, 30, 1.0),
    (2, dict(people=2, plateau=True), 0.1, 5, 30, 1.0),
    (3, dict(people=3, spread=0.7, tagnoise=0.3, clutter=5), 0.1, 5, 30, 1.0),
    (4, dict(people=4, clutter=8), 0.1, 3, 30, 1.0),
    (5, dict(people=5, spread=0.3, tagnoise=0.3), 0.1, 5, 30, 1.0),
    (6, dict(people=6, presence=0.6), 0.1, 5, 30, 0.5),
    (7, dict(people=4, c=14, h=32, w=64), 0.1, 5, 30, 1.0),
    (8, dict(people=8, presence=0.9), 0.1, 5, 8, 1.0),          # max_count clips the peak list and the persons
    (9, dict(people=3, clutter=12), 0.35, 7, 10, 2.0),
    (10, dict(people=0, clutter=3), 0.1, 5, 30, 1.0),
    (11, dict(people=2, h=16, w=16, n=3), 0.1, 1, 30, 1.0),      # window 1: every pixel >= threshold is a peak
]


def random_case(seed):
    """The randomised sweep (threshold 0.1, window 5, max_count 30, tag threshold 1.0, JOINT_ORDER_17) for seeds
    RANDOM_SEEDS; images may exceed the reference's 10-entry arrays, the checks skip those."""
    return make_case(seed, people=1 + seed % 6, spread=[2.0, 0.7, 0.3][seed % 3], tagnoise=[0.05, 0.3][seed % 2],
                     plateau=seed % 5 == 0, clutter=[0, 5, 12][seed % 3])


RANDOM_SEEDS = range(100, 160)
