"""CPU checks of the fast_utils oracle (SURVEY.md 8(f) row 2): the C restatement against golden vectors produced by the
reference's own native code (oracle/make_golden_fast_utils.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import fast_utils_cases as cases
from oracle import fast_utils_ref as fu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "fast_utils.npz")
GOLD_RANDOM = os.path.join(os.path.dirname(__file__), "golden", "fast_utils_random.npz")


def test_port_matches_golden():
    g = np.load(GOLD)
    for idx, (seed, kw, thr, win, m, tthr) in enumerate(cases.GOLDEN_CASES):
        det, tm = cases.make_case(seed, **kw)
        pre = "c%02d_" % idx
        count, val, tag, ind = fu.find_peaks(det, tm, thr, win, m, "port")
        for name, arr in (("count", count), ("val", val), ("tag", tag), ("ind", ind)):
            assert np.array_equal(arr, g[pre + name]), (idx, name)
        jo = cases.joint_order(det.shape[1])
        for i in range(det.shape[0]):
            num, ans, st = fu.assign(count[i], val[i], tag[i], ind[i], jo, tthr, m, "port")
            assert st == 0 and num == g[pre + "num"][i], (idx, i)
            assert np.array_equal(ans, g[pre + "ans"][i]), (idx, i)


def test_port_matches_compiled_reference():
    """the randomised sweep against what the reference's compiled code returned for it (tests/golden/fast_utils_random.npz)"""
    from oracle.make_golden import tensor_digest
    g = np.load(GOLD_RANDOM)
    checked = 0
    for seed in cases.RANDOM_SEEDS:
        det, tm = cases.random_case(seed)
        pre = "s%d_" % seed
        a = fu.find_peaks(det, tm, 0.1, 5, 30, "port")
        count, val, tag, ind = a
        assert np.array_equal(count, g[pre + "count"]), seed
        for name, arr in (("val", val), ("tag", tag), ("ind", ind)):
            assert tensor_digest(arr) == g[pre + name], (seed, name)
        for i in range(det.shape[0]):
            if count[i].max() > 10:
                continue
            n1, a1, s1 = fu.assign(count[i], val[i], tag[i], ind[i], cases.JOINT_ORDER_17, 1.0, 30, "port")
            if n1 > 10:      # the reference's [10] arrays would be overrun
                continue
            assert s1 == 0 and n1 == g[pre + "num"][i] and tensor_digest(a1) == g[pre + "ans"][i], (seed, i)
            checked += 1
    assert checked > 80


def test_port_beyond_reference_limit_terminates():
    det, tm = cases.make_case(7, people=20, clutter=30)
    count, val, tag, ind = fu.find_peaks(det, tm, 0.1, 5, 30, "port")
    assert count.max() > 10
    num, ans, st = fu.assign(count[0], val[0], tag[0], ind[0], cases.JOINT_ORDER_17, 1.0, 30, "port")
    assert st == 0 and 10 < num <= 30


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful without a CUDA device")
def test_plugin_mirror_has_no_cpu_fallback():
    from litepose_b200.fast_utils import plugins
    x = torch.zeros(1, 2, 8, 8)
    with pytest.raises(RuntimeError):
        plugins.find_peaks(x, x, 0.1, 5, 4)
