"""ORACLE - TEST INFRASTRUCTURE ONLY.  Generates tests/golden/fast_utils.npz (the listed cases) and
tests/golden/fast_utils_random.npz (the randomised sweep) from the reference's own native code compiled where it lies
(oracle/_ref/libfastutils_ref.so, recipe oracle/native/build_native.py).  Needs the reference checkout:
python -m oracle.make_golden_fast_utils"""
import os

import numpy as np

from . import fast_utils_cases as cases
from . import fast_utils_ref as fu
from .make_golden import tensor_digest
from .native import build_native


def main():
    built = build_native.build()
    assert "ref" in built, "the reference sources are not available here"
    out = {}
    for idx, (seed, kw, thr, win, m, tthr) in enumerate(cases.GOLDEN_CASES):
        det, tm = cases.make_case(seed, **kw)
        count, val, tag, ind = fu.find_peaks(det, tm, thr, win, m, "ref")
        assert count.max(initial=0) <= 10
        jo = cases.joint_order(det.shape[1])
        nums, anss = [], []
        for i in range(det.shape[0]):
            num, ans, _ = fu.assign(count[i], val[i], tag[i], ind[i], jo, tthr, m, "ref")
            assert num <= 10
            nums.append(num)
            anss.append(ans)
        pre = "c%02d_" % idx
        out[pre + "count"], out[pre + "val"], out[pre + "tag"], out[pre + "ind"] = count, val, tag, ind
        out[pre + "num"] = np.asarray(nums, np.int32)
        out[pre + "ans"] = np.stack(anss)
    gold = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
    path = os.path.join(gold, "fast_utils.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")
    out = {}
    for seed in cases.RANDOM_SEEDS:
        det, tm = cases.random_case(seed)
        count, val, tag, ind = fu.find_peaks(det, tm, 0.1, 5, 30, "ref")
        # num -1: an image the reference's 10-entry arrays cannot hold (more candidates, or more persons in the port);
        # the float arrays are stored as digests (the full sweep is a few hundred kB)
        nums, anss = [], []
        for i in range(det.shape[0]):
            num, ans = -1, np.zeros((30, det.shape[1], 4), np.float32)
            if count[i].max() <= 10:
                n1, _, _ = fu.assign(count[i], val[i], tag[i], ind[i], cases.JOINT_ORDER_17, 1.0, 30, "port")
                if n1 <= 10:
                    num, ans, _ = fu.assign(count[i], val[i], tag[i], ind[i], cases.JOINT_ORDER_17, 1.0, 30, "ref")
            nums.append(num)
            anss.append(tensor_digest(ans))
        pre = "s%d_" % seed
        out[pre + "count"] = count
        for name, arr in (("val", val), ("tag", tag), ("ind", ind)):
            out[pre + name] = np.array(tensor_digest(arr))
        out[pre + "num"] = np.asarray(nums, np.int32)
        out[pre + "ans"] = np.array(anss)
    path = os.path.join(gold, "fast_utils_random.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
