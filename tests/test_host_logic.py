"""CPU: C-ABI surface (every symbol the header declares is exported and bound), config
mirrors, drop-in module contract (state_dict keys, deepcopy, half wrapper on CPU), shard
logic, and the world_size-2 gloo gather."""
import copy
import ctypes
import os
import re
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from litepose_b200 import _lib, synth
from litepose_b200.config import FLIP_CONFIG, get_arch, get_cfg
from litepose_b200.dist import shard_range

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_c_abi_exports_match_header():
    hdr = open(os.path.join(ROOT, "include", "litepose_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(lp_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    lib = _lib.load()          # raises AttributeError if the .so lacks a bound symbol
    for name in declared:
        assert hasattr(lib, name), "header declares %s but the library does not export it" % name
        assert name in _lib.SIGNATURES, "ctypes binding missing for %s" % name
    assert set(_lib.SIGNATURES) == declared
    assert lib.lp_version() >= 100


def test_host_side_packers_and_errors():
    lib = _lib.load()
    assert lib.lp_pw1x1_packed_elems(16, 96) == 96 * 64
    assert lib.lp_pw1x1_packed_elems(120, 720) == 6 * 2 * 128 * 64     # 720 -> 6 chunks of 128 MMA columns
    assert lib.lp_pw1x1_packed_bias_elems(720) == 768
    assert lib.lp_pw1x1_packed_elems(48, 288) == 3 * 1 * 128 * 64      # 288 -> 3 chunks of 128
    assert lib.lp_pw1x1_packed_elems(120, 160) == 2 * 160 * 64          # <= 160: one chunk (fused kernel layout)
    assert lib.lp_pw1x1_packed_elems(32, 192) == 2 * 1 * 128 * 64       # 192 -> 128 + 64 (second chunk half empty)
    k, n = 24, 40
    w = (np.arange(n * k, dtype=np.float32).reshape(n, k) / 100).astype(np.float16).view(np.uint16)
    wp = np.zeros(lib.lp_pw1x1_packed_elems(k, n), np.uint16)
    bp = np.zeros(lib.lp_pw1x1_packed_bias_elems(n), np.float32)
    assert lib.lp_pw1x1_pack(w.ctypes.data, None, k, n, wp.ctypes.data, bp.ctypes.data) == 0
    t = wp.reshape(1, 1, 48, 64)
    assert np.array_equal(t[0, 0, :n, :k], w) and not t[0, 0, n:, :].any() and not t[0, 0, :, k:].any()
    assert lib.lp_pw1x1_pack(None, None, k, n, wp.ctypes.data, bp.ctypes.data) == 1
    assert b"lp_pw1x1_pack" in lib.lp_last_error()
    # deconv program: 9 shifts per 64-channel block, 16 (phase, tap) weight tiles per block
    assert lib.lp_deconv_packed_elems(120, 48, 32) == (2 + 1) * 16 * 32 * 64
    assert lib.lp_nms_topk_workspace_bytes(2, 14, 512, 512, 30) == 2 * 14 * 8 * 8 * 30 * 8 + 2 * 14 * 8   # bands x warps lists + thresholds


def test_round2_entry_points_validate_arguments():
    """Argument errors of the entry points added in round 2 are reported before anything touches a device (no GPU here):
    LP_ERR_BAD_ARG + a message naming the entry point."""
    lib = _lib.load()
    one = ctypes.c_void_p(16)      # never dereferenced: the checks fail first
    assert lib.lp_glue_scale_f32(None, one, None, None, None, 1, 14, 14, 0, 8, 8, 0, 16, 16, 0, 1.0, one, one, None) == 1
    assert b"lp_glue_scale_f32" in lib.lp_last_error()
    # model_joints < J, divide_by <= 0, a 10x shrink
    assert lib.lp_glue_scale_f32(one, one, None, None, None, 1, 14, 13, 0, 8, 8, 0, 16, 16, 0, 1.0, one, one, None) == 1
    assert b"model_joints" in lib.lp_last_error()
    assert lib.lp_glue_scale_f32(one, one, None, None, None, 1, 14, 14, 0, 8, 8, 0, 16, 16, 1, 0.0, one, None, None) == 1
    assert lib.lp_glue_scale_f32(one, one, None, None, None, 1, 14, 14, 0, 80, 80, 0, 16, 16, 0, 1.0, one, one, None) == 1
    assert b"shrinks" in lib.lp_last_error()
    assert lib.lp_glue_f32(one, one, None, None, None, 1, 14, 8, 8, 0, 16, 16, one, None, None) == 1      # tag required
    assert lib.lp_pack_payload_f32(one, one, one, 2, 420, 70, 421, one, None) == 1                         # keep > pcap
    assert b"lp_pack_payload_f32" in lib.lp_last_error()
    assert lib.lp_plant_crowd_f32(one, None, None, 5, one, None, None, 0, None) == 1                        # list without data
    assert lib.lp_plant_crowd_f32(one, None, None, 0, one, None, None, 0, None) == 0                        # nothing to plant
    assert lib.lp_tag_match_f32(one, one, one, 1, 14, 65, 2, 64, one, 0.1, 1.0, 1, 0, 65, 14 * 65, one, one, one, 1 << 30,
                                None) == 1
    assert b"K<=64" in lib.lp_last_error()
    assert lib.lp_tag_match_workspace_bytes(2, 14, 64, 2, 14 * 64) == 2 * 14 * 64 * (4 + 4 + 14 * 2 * 4)


def test_pipeline_cfg_validation_is_host_side():
    """LitePosePipeline._validate_cfg: what the fused glue covers and what it rejects (no GPU needed)."""
    from litepose_b200.pipeline import LitePosePipeline
    ok = get_cfg(input_size=128)
    ok.TEST.SCALE_FACTOR = [2, 1, 0.5]
    LitePosePipeline._validate_cfg(ok)
    ok.DATASET.WITH_CENTER, ok.MODEL.TAG_PER_JOINT = True, True
    LitePosePipeline._validate_cfg(ok)
    for bad_scales in ([0.5, 2], [1, 1], [0, 1]):
        c = get_cfg(input_size=128)
        c.TEST.SCALE_FACTOR = bad_scales
        with pytest.raises(ValueError):
            LitePosePipeline._validate_cfg(c)
    c = get_cfg(input_size=128)
    c.DATASET.WITH_CENTER, c.TEST.IGNORE_CENTER, c.MODEL.TAG_PER_JOINT = True, True, False
    with pytest.raises(NotImplementedError):
        LitePosePipeline._validate_cfg(c)
    c = get_cfg(input_size=128)
    c.LOSS.NUM_STAGES = 3
    with pytest.raises(NotImplementedError):
        LitePosePipeline._validate_cfg(c)


def test_config_mirrors_reference_values():
    cfg = get_cfg()
    assert cfg.DATASET.NUM_JOINTS == 14 and cfg.TEST.NMS_KERNEL == 5 and cfg.TEST.DETECTION_THRESHOLD == 0.1
    assert sorted(FLIP_CONFIG["CROWDPOSE"]) == list(range(14))
    assert get_arch("S")["deconv_setting"] == [32, 24, 32]


def test_dropin_module_contract():
    from litepose_b200.lib.models.pose_mobilenet import get_pose_net
    cfg = get_cfg(input_size=64)
    model = get_pose_net(cfg, True, get_arch("XS"))
    sd = model.state_dict()
    assert len(sd) == 679
    for k in ("first.0.0.weight", "stage.2.4.depth_conv.0.weight", "deconv_refined.0.weight",
              "deconv_bnrelu.0.0.running_mean", "final_raw.1.conv.3.weight"):
        assert k in sd
    assert model.channel == [16, 16, 32, 48, 80] and model.num_deconv_layers == 3
    m2 = copy.deepcopy(model)
    m2.load_state_dict(sd, strict=True)
    model.eval()
    x = synth.make_frames(1, 64, seed=1)
    with torch.no_grad():
        o = model(x)                  # CPU tensor: module graph (the valid.py:147-150 summary call)
    assert [tuple(t.shape) for t in o] == [(1, 28, 16, 16), (1, 14, 32, 32)]
    half = torch.nn.Sequential(m2.half())
    assert next(half.parameters()).dtype == torch.float16


def test_engine_cache_signature_tracks_weight_updates():
    """The packed-weight cache key (ADVICE round 1: stale engine after in-place updates) changes with every in-place
    update, re-assignment and load, and with nothing else."""
    from litepose_b200.lib.models.pose_mobilenet import get_pose_net
    model = get_pose_net(get_cfg(input_size=64), False, get_arch("XS")).eval()
    s0 = model._lp_signature()
    assert model._lp_signature() == s0
    with torch.no_grad():
        model(synth.make_frames(1, 64, seed=1))          # an eval forward touches nothing
    assert model._lp_signature() == s0
    with torch.no_grad():
        model.first[0][0].weight.mul_(1.5)               # optimizer-style in-place update
    s1 = model._lp_signature()
    assert s1 != s0
    model.first[3].running_mean.add_(0.1)                # BN statistics
    s2 = model._lp_signature()
    assert s2 != s1
    model.first[2].weight = torch.nn.Parameter(model.first[2].weight.detach().clone())   # re-assignment
    assert model._lp_signature() != s2
    sd = copy.deepcopy(model.state_dict())
    s3 = model._lp_signature()
    model.load_state_dict(sd)
    assert model._lp_signature() != s3
    assert copy.deepcopy(model)._lp_cache is not model._lp_cache
    # writes through ``.data`` have their own version counter: documented as needing lp_invalidate()
    s4 = model._lp_signature()
    model.first[3].running_mean.data.add_(0.1)
    assert model._lp_signature() == s4
    model.lp_invalidate()
    assert not model._lp_cache.engines


def test_shard_range():
    assert [shard_range(256, r, 8) for r in range(8)] == [(32 * r, 32 * r + 32) for r in range(8)]
    parts = [shard_range(10, r, 4) for r in range(4)]
    assert parts == [(0, 3), (3, 6), (6, 8), (8, 10)]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, q):
    import torch.distributed as dist
    from litepose_b200.dist import gather_packed, shard_range
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lo, hi = shard_range(5, rank, world)
    packed = torch.arange(lo, hi, dtype=torch.float32).view(-1, 1).repeat(1, 7) + 0.5
    out = gather_packed(packed, dst=0)
    if rank == 0:
        q.put(torch.cat(out, 0).numpy())
    else:
        assert out is None
    dist.destroy_process_group()


def test_gather_world2_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res.shape == (5, 7) and np.array_equal(res[:, 0], np.arange(5) + 0.5)


def test_folded_checkpoint_roundtrip(tmp_path):
    """SURVEY 8(f) row 4: the folded, kernel-packed checkpoint reproduces every array the engine prepared (CPU is
    enough for preparation; running needs CUDA and says so)."""
    import torch
    from litepose_b200.config import get_arch, get_cfg
    from litepose_b200.engine import LitePoseEngine
    from litepose_b200.lib.models.pose_mobilenet import get_pose_net
    from litepose_b200 import synth
    arch = get_arch("XS")
    torch.manual_seed(0)
    model = synth.randomize_bn_(get_pose_net(get_cfg(), False, arch), 1).eval()
    eng = LitePoseEngine(model.state_dict(), arch, "cpu")
    path = str(tmp_path / "xs.folded.npz")
    eng.export_folded(path)
    back = LitePoseEngine.from_folded(path, "cpu")

    def same(a, b, where=""):
        if isinstance(a, dict):
            assert set(a) == set(b), where
            for k in a:
                same(a[k], b[k], where + "/" + str(k))
        elif isinstance(a, list):
            assert len(a) == len(b), where
            for i, (x, y) in enumerate(zip(a, b)):
                same(x, y, where + "/%d" % i)
        elif torch.is_tensor(a):
            assert a.dtype == b.dtype and torch.equal(a, b), where
        else:
            assert a == b, where

    same(eng.P, back.P)
    assert back.channels == eng.channels and back.arch == arch
    with pytest.raises(RuntimeError):
        back.run(torch.zeros(1, 3, 64, 64))


def test_block_and_stem_host_helpers():
    """host-only entry points of the round-2 kernels (no GPU needed): shape admission and weight packing"""
    import numpy as np
    from litepose_b200 import _lib
    lib = _lib.load()
    # LitePose-S: stages 0-2 fit the block kernel (stage 2 in streaming mode), stage 3 (Cin = 120) does not
    assert [lib.lp_block_s1_supported(*c) for c in ((16, 96, 16), (32, 192, 32), (48, 288, 48), (120, 720, 120), (48, 288, 120))] \
        == [1, 1, 1, 0, 0]
    assert lib.lp_block_s1_supported(12, 72, 16) == 0 and lib.lp_block_s1_supported(16, 96, 20) == 0     # multiples of 8
    assert lib.lp_stem_fused_supported(512, 512, 16) == 1 and lib.lp_stem_fused_supported(512, 510, 16) == 0
    assert lib.lp_stem_fused_supported(640, 640, 24) == 1 and lib.lp_stem_fused_supported(64, 64, 40) == 0
    cin, ce = 24, 80
    w = (np.arange(ce * cin, dtype=np.uint16).reshape(ce, cin) + 1)
    out = np.full(lib.lp_block_s1_wexp_elems(cin, ce), 0xffff, np.uint16)
    assert out.size == 96 * 64                      # 3 slabs of 32 rows, K padded to 64
    _lib.check(lib.lp_block_s1_pack_wexp(w.ctypes.data, cin, ce, out.ctypes.data))
    out = out.reshape(96, 64)
    assert np.array_equal(out[:ce, :cin], w) and not out[:ce, cin:].any() and not out[ce:].any()


def test_dropin_install_refuses_late_binding(tmp_path):
    """litepose_b200.dropin.install() must raise when a reference package of the same name is already imported"""
    import subprocess
    import sys
    pkg = tmp_path / "models"
    pkg.mkdir()
    (pkg / "__init__.py").write_text("x = 1\n")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import models; import litepose_b200.dropin as d\n"
            "try:\n    d.install()\nexcept ImportError as e:\n    print('refused', 'models' in str(e))\n" % (ROOT, str(tmp_path)))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert "refused True" in r.stdout, r.stdout + r.stderr


def test_load_experiment_without_yacs(tmp_path):
    """config.load_experiment: the reference's --cfg / --superconfig / opts flow (valid.py:95-111) on an experiment file
    in the reference's format; the evaluation keys equal get_cfg()'s literal table."""
    from litepose_b200.config import load_experiment
    text = """
DATASET: {DATASET: crowd_pose_kpt, DATASET_TEST: crowd_pose, INPUT_SIZE: 256, OUTPUT_SIZE: [64, 128], MAX_NUM_PEOPLE: 30, NUM_JOINTS: 14}
LOSS: {NUM_STAGES: 2, WITH_AE_LOSS: [True, False], WITH_HEATMAPS_LOSS: [True, True]}
MODEL:
  NAME: pose_mobilenet
  NUM_JOINTS: 14
  TAG_PER_JOINT: True
  EXTRA: {FINAL_CONV_KERNEL: 1, NUM_DECONV_LAYERS: 3, NUM_DECONV_FILTERS: [64, 48, 32], NUM_DECONV_KERNELS: [4, 4, 4]}
TEST:
  FLIP_TEST: True
  IMAGES_PER_GPU: 1
  SCALE_FACTOR: [1]
  DETECTION_THRESHOLD: 0.1
  WITH_HEATMAPS: (True, True)
  WITH_AE: (True, False)
  PROJECT2IMAGE: True
  NMS_KERNEL: 5
  NMS_PADDING: 2
TRAIN: {LR: 4e-3, WD: 1e-4}
"""
    path = tmp_path / "mobile.yaml"
    path.write_text(text)
    cfg, arch = load_experiment(str(path), superconfig="S")
    ref = get_cfg(input_size=448)
    assert arch["deconv_setting"] == [32, 24, 32] and cfg.DATASET.INPUT_SIZE == 448 and cfg.DATASET.OUTPUT_SIZE == [112, 224]
    assert cfg.TEST.WITH_HEATMAPS == (True, True) and cfg.TEST.WITH_AE == (True, False) and cfg.TRAIN.WD == 1e-4
    skip = {"INIT_WEIGHTS"}          # get_cfg() builds random-init models (no checkpoint in the synthetic setting)
    for sec in ("MODEL", "LOSS", "DATASET", "TEST"):
        for k, v in ref[sec].items():
            if k in skip:
                continue
            got = cfg[sec][k]
            if isinstance(v, (list, tuple)):
                assert list(got) == list(v), (sec, k)
            elif isinstance(v, dict):
                assert dict(got) == dict(v), (sec, k)
            else:
                assert got == v, (sec, k, got, v)
    # opts + the WITH_CENTER adjustment of update_config (lib/config/default.py:175-177)
    cfg2, _ = load_experiment(str(path), opts=["DATASET.WITH_CENTER", "True", "TEST.SCALE_FACTOR", "[0.5, 1, 2]"])
    assert cfg2.DATASET.NUM_JOINTS == 15 and cfg2.MODEL.NUM_JOINTS == 15 and cfg2.TEST.SCALE_FACTOR == [0.5, 1, 2]
    with pytest.raises(KeyError):
        load_experiment(str(path), opts=["TEST.NO_SUCH_KEY", "1"])
    # the reference's own experiment file (experiments/crowd_pose/mobilenet/mobile.yaml, stored verbatim)
    cfg3, _ = load_experiment(os.path.join(ROOT, "tests", "golden", "crowd_pose_mobile.yaml"), superconfig="S")
    for sec in ("MODEL", "LOSS", "DATASET", "TEST"):
        for k, v in ref[sec].items():
            if k in skip:
                continue
            got = cfg3[sec][k]
            if isinstance(v, (list, tuple)):
                assert list(got) == list(v), (sec, k)
            elif isinstance(v, dict):        # the file may carry more keys (PRETRAINED_LAYERS ...)
                assert all(list(got[k2]) == list(v2) if isinstance(v2, list) else got[k2] == v2 for k2, v2 in v.items()), (sec, k)
            else:
                assert got == v, (sec, k)


def test_valid_synthetic_cli_dry_run(tmp_path):
    """tools/valid_synthetic.py takes valid.py's arguments (--cfg, --superconfig, KEY VALUE opts) and resolves them as
    valid.py:95-111 does; --dry-run stops before the first CUDA call."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("valid_synthetic", os.path.join(ROOT, "tools", "valid_synthetic.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    path = tmp_path / "exp.yaml"
    path.write_text("DATASET: {DATASET: crowd_pose_kpt, DATASET_TEST: crowd_pose, NUM_JOINTS: 14}\n"
                    "MODEL: {NAME: pose_mobilenet, NUM_JOINTS: 14, EXTRA: {NUM_DECONV_LAYERS: 3, NUM_DECONV_KERNELS: [4, 4, 4]}}\n"
                    "LOSS: {NUM_STAGES: 2, WITH_AE_LOSS: [True, False], WITH_HEATMAPS_LOSS: [True, True]}\n"
                    "TEST:\n  FLIP_TEST: True\n  WITH_HEATMAPS: (True, True)\n  WITH_AE: (True, False)\n  PROJECT2IMAGE: True\n")
    out = mod.main(["--cfg", str(path), "--superconfig", "XS", "--dry-run", "TEST.SCALE_FACTOR", "[0.5, 1]"])
    assert out["input_size"] == 256 and out["scale_factor"] == [0.5, 1] and out["flip_test"] is True
    with pytest.raises(ValueError):            # the reference needs the scale-1 pass (valid.py:224)
        mod.main(["--cfg", str(path), "--superconfig", "XS", "--dry-run", "TEST.SCALE_FACTOR", "[0.5, 2]"])
