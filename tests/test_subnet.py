"""SURVEY 8(f) row 4: sub-network extraction from a larger checkpoint (reference weight_transfer.py:75-146)."""
import os

import numpy as np
import pytest
import torch

from litepose_b200.config import get_arch, get_cfg
from litepose_b200.lib.models.pose_mobilenet import get_pose_net
from litepose_b200.subnet import extract_subnet, extract_subnet_state_dict

GOLD = os.path.join(os.path.dirname(__file__), "golden", "subnet_transfer.npz")


def _big(seed=0):
    torch.manual_seed(seed)
    net = get_pose_net(get_cfg(), False, get_arch("L"))
    for m in net.modules():                                      # non-trivial BN statistics
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_(0, 0.1)
            m.running_var.uniform_(0.75, 1.25)
    return net.eval()


@pytest.mark.parametrize("arch", ["XS", "S", "M"])
def test_prefix_slices_and_strict_load(arch):
    big = _big()
    sub = extract_subnet(big.state_dict(), get_cfg(), get_arch(arch))
    sd, sup = sub.state_dict(), big.state_dict()
    assert len(sd) == 679
    for k, v in sd.items():
        assert torch.equal(v, sup[k][tuple(slice(0, d) for d in v.shape)].to(v.dtype)), k
    # a '1.'-prefixed (network_to_half) checkpoint works too; too small a source is refused
    pref = {"1." + k: v for k, v in sup.items()}
    again = extract_subnet_state_dict(pref, sd)
    assert all(torch.equal(again[k], sd[k]) for k in sd)
    with pytest.raises(ValueError):
        extract_subnet_state_dict(sd, sup)


def test_matches_reference_transfer():
    """against the reference's own transfer() (weight_transfer.py) from the same LitePose-L into LitePose-S and a tiny
    arch: tests/golden/subnet_transfer.npz holds a digest of every tensor it produced (oracle/make_golden.py)"""
    from litepose_b200.synth import randomize_bn_
    from oracle.make_golden import SUBNET_TINY_ARCH, tensor_digest
    g = np.load(GOLD)
    cfg = get_cfg()
    torch.manual_seed(3)                               # the reference model's initialisation (oracle/refshim.py)
    big = randomize_bn_(get_pose_net(cfg, False, get_arch("L")), 1).eval().state_dict()
    for name, arch in (("S", get_arch("S")), ("tiny", SUBNET_TINY_ARCH)):
        keys = [str(k) for k in g[name + "_keys"]]
        want = dict(zip(keys, (str(d) for d in g[name + "_digest"])))
        torch.manual_seed(4)
        target = randomize_bn_(get_pose_net(cfg, False, arch), 1).eval().state_dict()
        assert list(target) == keys
        got = extract_subnet_state_dict(big, target)
        for k in keys:
            if k.endswith("num_batches_tracked"):
                continue                                   # the reference leaves the target's own counter
            assert tensor_digest(got[k]) == want[k], (name, k)
