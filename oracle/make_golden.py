"""ORACLE (test infrastructure, not product code).

Generate the committed known-answer fixtures under tests/golden/ by running the
UNMODIFIED reference (imported in place from /root/reference through
oracle/refshim.py) on seeded synthetic inputs.  The reference ships no golden
vectors or tests of its own (SURVEY.md §4), so these are the pins for both the
oracle restatements and the CUDA path.  Run in the build container only:

    python -m oracle.make_golden
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from litepose_b200 import synth  # noqa: E402
from litepose_b200.config import get_arch, get_cfg  # noqa: E402
from oracle import refshim  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

TINY_ARCH = {
    "img_size": 64, "input_channel": 16, "deconv_setting": [16, 24, 24],
    "backbone_setting": [
        {"num_blocks": 2, "stride": 2, "channel": 16, "block_setting": [[6, 7], [6, 7]]},
        {"num_blocks": 2, "stride": 2, "channel": 24, "block_setting": [[6, 7], [6, 7]]},
        {"num_blocks": 2, "stride": 2, "channel": 40, "block_setting": [[6, 7], [6, 7]]},
        {"num_blocks": 2, "stride": 1, "channel": 48, "block_setting": [[6, 7], [6, 7]]},
    ],
}


def sd_digest(sd):
    h = hashlib.sha256()
    for k in sd:
        h.update(k.encode())
        h.update(sd[k].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def tensor_digest(t):
    """sha256 over a tensor's or array's dtype, shape and bytes: equal digests <=> equal arrays (for finite values)."""
    a = t.detach().cpu().contiguous().numpy() if torch.is_tensor(t) else np.ascontiguousarray(t)
    h = hashlib.sha256()
    h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


# the second target of the sub-network transfer check (besides LitePose-S): three stages deep, one block in the last
SUBNET_TINY_ARCH = {
    "img_size": 256, "input_channel": 16, "deconv_setting": [16, 24, 24],
    "backbone_setting": [{"num_blocks": 2, "stride": 2, "channel": 16, "block_setting": [[6, 7]] * 2},
                         {"num_blocks": 3, "stride": 2, "channel": 24, "block_setting": [[6, 7]] * 3},
                         {"num_blocks": 2, "stride": 2, "channel": 40, "block_setting": [[6, 7]] * 2},
                         {"num_blocks": 1, "stride": 1, "channel": 64, "block_setting": [[6, 7]] * 1}]}


def golden_subnet_transfer():
    """The reference's own transfer() (weight_transfer.py, function bodies executed where the file lies) from a
    LitePose-L (seed 3) into LitePose-S and SUBNET_TINY_ARCH (seed 4): one digest per tensor of the target's state
    dict (the full tensors are tens of MB)."""
    import ast
    path = os.path.join(refshim.REF_ROOT, "weight_transfer.py")
    fns = [n for n in ast.parse(open(path).read()).body if isinstance(n, ast.FunctionDef) and n.name.startswith("transfer")]
    cfg = get_cfg()
    ns = {"cfg": cfg}
    exec(compile(ast.Module(body=fns, type_ignores=[]), "weight_transfer_fns", "exec"), ns)
    big = refshim.build_reference_model(cfg, get_arch("L"), seed=3)
    blob = {}
    for name, arch in (("S", get_arch("S")), ("tiny", SUBNET_TINY_ARCH)):
        small = refshim.build_reference_model(cfg, arch, seed=4)
        ns["transfer"](big, small, arch)
        want = small.state_dict()
        blob[name + "_keys"] = np.array(list(want))
        blob[name + "_digest"] = np.array([tensor_digest(v) for v in want.values()])
    np.savez_compressed(os.path.join(OUT, "subnet_transfer.npz"), **blob)


def golden_model():
    ns = refshim.load()
    # (1) tiny arch: weights + per-layer activations committed
    cfg = get_cfg(input_size=64)
    model = refshim.build_reference_model(cfg, TINY_ARCH)
    sd = model.state_dict()
    x = synth.make_frames(2, 64, seed=7)
    acts = {}
    hooks = []
    names = ["first.0", "first.1", "first", "stage.0.0.inv", "stage.0.0.depth_conv", "stage.0.0",
             "stage.0.1", "stage.1.0", "stage.2.1", "stage.3.1", "deconv_bnrelu.0", "deconv_bnrelu.1",
             "deconv_bnrelu.2", "final_refined.0.conv.2", "final_raw.1.conv.2"]
    mods = dict(model.named_modules())
    for nme in names:
        hooks.append(mods[nme].register_forward_hook(
            lambda m, i, o, nme=nme: acts.__setitem__(nme, o.detach().clone())))
    with torch.no_grad():
        outs = model(x)
    for h in hooks:
        h.remove()
    blob = {"x": x.numpy(), "out0": outs[0].numpy(), "out1": outs[1].numpy()}
    for k, v in sd.items():
        blob["sd/" + k] = v.numpy()
    for k, v in acts.items():
        blob["act/" + k] = v.numpy()
    np.savez_compressed(os.path.join(OUT, "model_tiny.npz"), **blob)

    # (2) shipped archs with seeded weights: digest + outputs only
    for name, size in (("XS", 128), ("S", 128)):
        cfg = get_cfg(input_size=size)
        arch = get_arch(name)
        model = refshim.build_reference_model(cfg, arch)
        x = synth.make_frames(1, size, seed=11)
        with torch.no_grad():
            outs = model(x)
            half = ns.fp16util.network_to_half(refshim.build_reference_model(cfg, arch))
            outs_h = half(x)
        np.savez_compressed(
            os.path.join(OUT, "model_%s_%d.npz" % (name, size)),
            digest=np.array(sd_digest(model.state_dict())),
            out0=outs[0].numpy(), out1=outs[1].numpy(),
            out0_fp16eager=outs_h[0].numpy(), out1_fp16eager=outs_h[1].numpy())


def golden_glue():
    ns = refshim.load()
    g = torch.Generator().manual_seed(21)
    for flip, proj in ((True, True), (False, True), (True, False)):
        cfg = get_cfg(input_size=64, flip_test=flip, project2image=proj)
        a0 = torch.randn(2, 28, 16, 16, generator=g)
        a1 = torch.randn(2, 14, 32, 32, generator=g)
        b0 = torch.randn(2, 28, 16, 16, generator=g)
        b1 = torch.randn(2, 14, 32, 32, generator=g)
        calls = []

        def fake_model(img):
            calls.append(1)
            return [a0.clone(), a1.clone()] if len(calls) == 1 else [b0.clone(), b1.clone()]

        img = torch.zeros(2, 3, 64, 64)
        _, h, t = ns.inference.get_multi_stage_outputs(cfg, fake_model, img, flip, proj, (64, 64))
        fh, tl = ns.inference.aggregate_results(cfg, 1, None, [], h, t)
        tags = torch.cat(tl, dim=4)
        np.savez_compressed(os.path.join(OUT, "glue_flip%d_proj%d.npz" % (flip, proj)),
                            a0=a0.numpy(), a1=a1.numpy(), b0=b0.numpy(), b1=b1.numpy(),
                            final_heatmaps=fh.numpy(), tags=tags.numpy())


MULTISCALE_CASES = [
    # name, SCALE_FACTOR, PROJECT2IMAGE, FLIP_TEST, input_size (square images), seed
    ("ms_1_2_proj1", [1, 2], True, True, 64, 41),
    ("ms_05_1_proj0", [0.5, 1], False, True, 128, 42),
]


class FakeScaleModel(object):
    """Seeded random network outputs shaped by the image it is given: [N,2J,H/4,W/4], [N,J,H/2,W/2]; ``log`` keeps
    every call's outputs in call order (largest scale first, plain pass then mirrored pass)."""

    def __init__(self, nj, seed, tag_channels=None):
        self.nj, self.g, self.log = nj, torch.Generator().manual_seed(seed), []
        self.nt = nj if tag_channels is None else tag_channels

    def __call__(self, img):
        n, _, h, w = img.shape
        outs = [torch.randn(n, self.nj + self.nt, h // 4, w // 4, generator=self.g),
                torch.randn(n, self.nj, h // 2, w // 2, generator=self.g)]
        self.log.append(outs)
        return [o.clone() for o in outs]


def multiscale_inputs(cfg, size):
    """valid.py:198-212 for a square ``size`` x ``size`` image: base_size and the (empty) resized image per scale."""
    from litepose_b200.lib.utils.transforms import get_multi_scale_size
    img = np.zeros((size, size, 3), np.uint8)
    smin = min(cfg.TEST.SCALE_FACTOR)
    base, _, _ = get_multi_scale_size(img, cfg.DATASET.INPUT_SIZE, 1.0, smin)
    images = {}
    for s in cfg.TEST.SCALE_FACTOR:
        (w, h), _, _ = get_multi_scale_size(img, cfg.DATASET.INPUT_SIZE, s, smin)
        images[s] = torch.zeros(1, 3, h, w)
    return base, images


def golden_glue_multiscale():
    """The multi-scale loop of valid.py:205-225 run with the reference's own get_multi_stage_outputs / aggregate_results
    on a seeded fake model; inputs are reproduced from the seed in the tests (digest stored)."""
    ns = refshim.load()
    for name, scales, proj, flip, size, seed in MULTISCALE_CASES:
        cfg = get_cfg(input_size=size, flip_test=flip, project2image=proj)
        cfg.TEST.SCALE_FACTOR = list(scales)
        base, images = multiscale_inputs(cfg, size)
        fake = FakeScaleModel(cfg.DATASET.NUM_JOINTS, seed)
        final, tags_list = None, []
        for s in sorted(cfg.TEST.SCALE_FACTOR, reverse=True):
            _, h, t = ns.inference.get_multi_stage_outputs(cfg, fake, images[s], flip, proj, base)
            final, tags_list = ns.inference.aggregate_results(cfg, s, final, tags_list, h, t)
        final = final / float(len(cfg.TEST.SCALE_FACTOR))
        tags = torch.cat(tags_list, dim=4)
        dig = hashlib.sha256(b"".join(o.numpy().tobytes() for outs in fake.log for o in outs)).hexdigest()
        np.savez_compressed(os.path.join(OUT, "glue_%s.npz" % name), in_digest=np.array(dig),
                            final_heatmaps=final.numpy(), tags=tags.numpy())


GLUE_CFG_CASES = [
    # name, WITH_CENTER, IGNORE_CENTER, TAG_PER_JOINT, PROJECT2IMAGE, seed
    ("center_ignored", True, True, True, True, 51),
    ("center_kept", True, False, True, True, 52),
    ("shared_tag", False, True, False, True, 53),
    ("shared_tag_noproj", False, True, False, False, 54),
]


GLUE_CFG_SIZE = 32        # fake "image" side of the cfg-branch cases (the fake model only looks at the shape)


def glue_cfg(with_center, ignore_center, tag_per_joint, proj, size=64, dataset="crowd_pose"):
    """cfg as lib/config/default.py:175-177 leaves it: NUM_JOINTS counts the centre joint when WITH_CENTER is on"""
    cfg = get_cfg(dataset=dataset, input_size=size, flip_test=True, project2image=proj)
    cfg.DATASET.WITH_CENTER = with_center
    if with_center:
        cfg.DATASET.NUM_JOINTS += 1
        cfg.MODEL.NUM_JOINTS = cfg.DATASET.NUM_JOINTS
    cfg.TEST.IGNORE_CENTER = ignore_center
    cfg.MODEL.TAG_PER_JOINT = tag_per_joint
    return cfg


def golden_glue_cfgs():
    """get_multi_stage_outputs + aggregate_results of the unmodified reference for the cfg branches beyond the shipped
    mobile.yaml: WITH_CENTER (kept / ignored) and TAG_PER_JOINT off; seeded fake model, inputs reproduced in the tests."""
    ns = refshim.load()
    for name, center, ignore, per_joint, proj, seed in GLUE_CFG_CASES:
        cfg = glue_cfg(center, ignore, per_joint, proj)
        jm = cfg.DATASET.NUM_JOINTS
        fake = FakeScaleModel(jm, seed, None if per_joint else 1)
        img = torch.zeros(2, 3, GLUE_CFG_SIZE, GLUE_CFG_SIZE)
        _, h, t = ns.inference.get_multi_stage_outputs(cfg, fake, img, True, proj, (GLUE_CFG_SIZE, GLUE_CFG_SIZE))
        fh, tl = ns.inference.aggregate_results(cfg, 1, None, [], h, t)
        tags = torch.cat(tl, dim=4)
        dig = hashlib.sha256(b"".join(o.numpy().tobytes() for outs in fake.log for o in outs)).hexdigest()
        np.savez_compressed(os.path.join(OUT, "glue_cfg_%s.npz" % name), in_digest=np.array(dig),
                            final_heatmaps=fh.numpy(), tags=tags.numpy())


PARSER_CASES = [
    # name, J-dataset, h, w, T, people, seed
    ("p5_128_t2", "crowd_pose", 128, 128, 2, 5, 0),
    ("p5_128_t1", "crowd_pose", 128, 128, 1, 5, 1),
    ("p30_256_t2", "crowd_pose", 256, 256, 2, 30, 2),
    ("p3_64x96_t2", "crowd_pose", 64, 96, 2, 3, 3),
    ("p0_128_t2", "crowd_pose", 128, 128, 2, 0, 4),
    ("p12_256_t2", "crowd_pose", 256, 256, 2, 12, 5),
    ("p30_256_t1", "crowd_pose", 256, 256, 1, 30, 6),
    ("coco_p8_128_t2", "coco", 128, 160, 2, 8, 7),
    # the bench geometries (BASELINE configs 3 and 5): 512^2 with 5 persons, 640^2 with a 30-person crowd
    ("p5_512_t2", "crowd_pose", 512, 512, 2, 5, 8),
    ("p30_640_t2", "crowd_pose", 640, 640, 2, 30, 9),
]


def golden_parser(only=None):
    ns = refshim.load()
    for name, ds, h, w, t, people, seed in PARSER_CASES:
        if only and name not in only:
            continue
        cfg = get_cfg(dataset=ds, input_size=256)
        nj = cfg.DATASET.NUM_JOINTS
        det, tag = synth.plant_crowd(nj, h, w, t, num_people=people, seed=seed)
        dt = torch.from_numpy(det)[None]
        tt = torch.from_numpy(tag)[None]
        rp = ns.group.HeatmapParser(cfg)
        top = rp.top_k(dt, tt)
        blob = {"in_digest": np.array(hashlib.sha256(det.tobytes() + tag.tobytes()).hexdigest()),
                "val_k": top["val_k"], "loc_k": top["loc_k"], "tag_k": top["tag_k"]}
        for adj, ref in ((True, True), (True, False), (False, False)):
            ans, scores = rp.parse(dt.clone(), tt.clone(), adj, ref)
            a = np.array(ans[0], dtype=np.float32).reshape(-1, nj, 3 + t)
            blob["ans_a%d_r%d" % (adj, ref)] = a
            blob["scores_a%d_r%d" % (adj, ref)] = np.array(scores, dtype=np.float32)
        np.savez_compressed(os.path.join(OUT, "parser_%s.npz" % name), **blob)


def shared_tag_case(nj, h, w, t, people, seed):
    """Inputs of the MODEL.TAG_PER_JOINT=False case: the planted crowd with ONE tag map shared by all joints (every pixel
    takes the tag of the joint plane with the largest heat there)."""
    det, tag = synth.plant_crowd(nj, h, w, t, num_people=people, seed=seed)
    pick = det.argmax(axis=0)[None, :, :, None]
    shared = np.take_along_axis(tag, np.broadcast_to(pick, (1, h, w, t)), axis=0)
    return det, np.ascontiguousarray(shared)


def golden_parser_shared_tag():
    """lib/core/group.py:150-152 (TAG_PER_JOINT=False).  With refine the reference stops on an unassigned name
    (group.py:283-286) as soon as one person is found - recorded here, so only refine=False outputs exist."""
    ns = refshim.load()
    cfg = get_cfg(input_size=256)
    cfg.MODEL.TAG_PER_JOINT = False
    nj = cfg.DATASET.NUM_JOINTS
    det, tag = shared_tag_case(nj, 128, 160, 2, 6, 31)
    dt, tt = torch.from_numpy(det)[None], torch.from_numpy(tag)[None]
    rp = ns.group.HeatmapParser(cfg)
    top = rp.top_k(dt, tt)
    blob = {"in_digest": np.array(hashlib.sha256(det.tobytes() + tag.tobytes()).hexdigest()),
            "val_k": top["val_k"], "loc_k": top["loc_k"], "tag_k": top["tag_k"]}
    for adj in (True, False):
        ans, scores = rp.parse(dt.clone(), tt.clone(), adj, False)
        blob["ans_a%d_r0" % adj] = np.array(ans[0], dtype=np.float32).reshape(-1, nj, 5)
        blob["scores_a%d_r0" % adj] = np.array(scores, dtype=np.float32)
    try:
        rp.parse(dt.clone(), tt.clone(), True, True)
        blob["refine_raises"] = np.array("")
    except NameError as e:
        blob["refine_raises"] = np.array("NameError: %s" % e)
    np.savez_compressed(os.path.join(OUT, "parser_shared_tag_p6.npz"), **blob)


def golden_munkres():
    """Self-pinned restatement outputs on degenerate matrices (parity unpinned vs
    PyPI munkres, see oracle/munkres_ref.py) + the reference's own cost recipe."""
    from oracle.munkres_ref import Munkres
    rng = np.random.RandomState(5)
    mats, sols = [], []
    for trial in range(40):
        r = rng.randint(1, 13)
        c = rng.randint(1, 13)
        dist = rng.choice([0.0, 0.0, 0.0, 1.0, 2.0, 4.0], size=(r, c))
        val = rng.uniform(0.1, 1.0, size=(r, 1)).astype(np.float32).astype(np.float64)
        m = np.round(dist) * 100 - val
        if r > c:
            m = np.concatenate((m, np.zeros((r, r - c)) + 1e10), axis=1)
        pairs = Munkres().compute(m.copy())
        full = np.full((12, 12), np.nan)
        full[:m.shape[0], :m.shape[1]] = m
        sol = np.full((12, 2), -1, np.int32)
        sol[:len(pairs)] = np.array(pairs, np.int32).reshape(-1, 2)
        mats.append(full)
        sols.append(sol)
    np.savez_compressed(os.path.join(OUT, "munkres_cases.npz"), mats=np.stack(mats), sols=np.stack(sols))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    if len(sys.argv) > 2 and sys.argv[1] == "--parser-only":       # regenerate selected parser cases only
        golden_parser(only=set(sys.argv[2:]))
    elif len(sys.argv) > 1 and sys.argv[1] == "--new-r2":          # fixtures added in round 2 (others untouched)
        golden_parser_shared_tag()
        golden_glue_multiscale()
        golden_glue_cfgs()
    elif len(sys.argv) > 1 and sys.argv[1] == "--subnet-transfer":
        golden_subnet_transfer()
    else:
        golden_model()
        golden_glue()
        golden_parser()
        golden_parser_shared_tag()
        golden_glue_multiscale()
        golden_glue_cfgs()
        golden_munkres()
        golden_subnet_transfer()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
