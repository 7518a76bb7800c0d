#!/usr/bin/env python
"""Benchmark of the LitePose inference hot path (BASELINE.json metric):

    frames/sec, LitePose-S 512x512 end-to-end (backbone x2 with flip + glue + group), fp16, batch 32 per GPU.

    python bench.py --gpus N --steps K --warmup W            # sm_100a path (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host CPU cores

A "step" is one pass of the hot path over one batch of synthetic frames per GPU.  `value` is the
whole-job throughput with the frames resident in HBM; `e2e` is the same metric through the public
pipeline call with pinned HOST frames (H2D + result D2H inside the timed region, NCCL gather of the
packed keypoints when N > 1).  Timing: CUDA events on the launching stream, barrier + synchronize on
both sides, max over ranks.  Per-step working set (~2 GB of heat/tag maps at batch 32) exceeds the
126 MB L2, so no explicit flush is needed for the step timing; the single-kernel roofline timing
flushes L2 between iterations.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "frames/sec LitePose-S 512x512 end-to-end (backbone+group)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--arch", default="S")
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--batch", type=int, default=32, help="frames per GPU per step")
    ap.add_argument("--people", type=int, default=5)
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--ref-frames", type=int, default=2, help="frames per step of the CPU reference arm")
    ap.add_argument("--cpu-sample", type=int, default=48, help="frames of the cpu_baseline sample (b200 arm)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the packed keypoint payloads of the last timed step (device-resident and end-to-end) "
                         "to DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 path")
    return args


def payload_as_received(packed, keep):
    """Packed payload rows [..., keep*row + keep + 1] with the person slots beyond each image's count zeroed: the parser
    leaves them unwritten and LitePosePipeline.unpack() never reads them."""
    import numpy as np
    a = np.array(packed, dtype=np.float32)
    row = (a.shape[-1] - 1 - keep) // keep
    for r in a.reshape(-1, a.shape[-1]):
        p = min(int(r[-1]), keep)
        r[p * row:keep * row] = 0
        r[keep * row + p:keep * row + keep] = 0
    return a


def dump_outputs(directory, arrays):
    """One float32 .npy per array: the same arguments give the same inputs, so two builds compare output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def workload_config(args, n_gpus):
    return {
        "workload": "LitePose-%s %dx%d fp16 batch=%d/GPU: 2 forward passes (flip test) + fused glue "
                    "(PROJECT2IMAGE) + HeatmapParser NMS/top-K/tag-match/adjust/refine, %d planted persons/frame"
                    % (args.arch, args.size, args.size, args.batch, args.people),
        "arch": "search-%s.json" % args.arch, "input": [args.size, args.size], "batch_per_gpu": args.batch,
        "global_batch": args.batch * n_gpus, "eval_cfg": "experiments/crowd_pose/mobilenet/mobile.yaml",
        "parallelism": "dp%d (batch sharded, one NCCL gather of packed keypoints)" % n_gpus,
        "l2": "working set per step > L2 (no flush needed); roofline kernel timed with explicit L2 flush",
    }


# ------------------------------------------------------------------------------ clocks
class ClockSampler(object):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------ CPU arm (oracle port)
def cpu_reference_setup(args):
    import torch
    from litepose_b200 import synth
    from litepose_b200.config import get_arch, get_cfg
    from litepose_b200.lib.models.pose_mobilenet import get_pose_net
    from litepose_b200.pipeline import PlantedCrowd
    cfg = get_cfg(input_size=args.size)
    arch = get_arch(args.arch)
    torch.manual_seed(0)
    model = synth.scale_heads_(synth.randomize_bn_(get_pose_net(cfg, False, arch), 1)).eval()
    sd = {k: v.float() for k, v in model.state_dict().items()}
    # all the host threads the CPU path can USE: eager CPU convolutions at batch 1-2 slow down when
    # oversubscribed (128 threads measured 60x slower than 8 on the bench box), so probe a few counts
    from oracle import model_ref
    ncpu = os.cpu_count() or 1
    probe = synth.make_frames(1, args.size, seed=5)
    best, best_t = ncpu, None
    for nt in sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu}):
        torch.set_num_threads(nt)
        with torch.no_grad():
            model_ref.forward(sd, arch, probe)
            t0 = time.perf_counter()
            model_ref.forward(sd, arch, probe)
            dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = nt, dt
    torch.set_num_threads(best)
    return cfg, arch, sd


def cpu_reference_step(cfg, arch, sd, frames, plant):
    """The reference algorithm for the path on the host: fp32 eager forward x2 (flip), glue,
    planted persons, HeatmapParser.parse per image (oracle restatement; the Python reference itself
    cannot travel to the GPU box)."""
    import numpy as np
    import torch
    from oracle import glue_ref, group_ref, model_ref
    size = frames.shape[2]
    with torch.no_grad():
        _, hm, tg = glue_ref.multi_stage_outputs(cfg, lambda im: model_ref.forward(sd, arch, im), frames, True, True,
                                                 (frames.shape[3], size))
        det, tag = glue_ref.aggregate(cfg, hm, tg)
        det, tag = det.contiguous(), tag.contiguous()
        plant.apply(det, tag)
    parser = group_ref.HeatmapParser(cfg)
    out = []
    dn, tn = det.numpy(), tag.numpy()
    for i in range(frames.shape[0]):
        out.append(parser.parse(dn[i:i + 1], tn[i:i + 1], True, True))
    return out


_RESULT_FD = None


def claim_stdout():
    """stdout carries exactly ONE line, the JSON result.  Libraries print there too (NCCL announces its version on the
    first communicator, cuDNN / torch warnings ...), so fd 1 is pointed at stderr for the life of the process and the
    result line is written to a private duplicate of the original stdout."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from litepose_b200 import synth
    from litepose_b200.pipeline import PlantedCrowd
    cfg, arch, sd = cpu_reference_setup(args)
    nf = args.ref_frames
    frames = synth.make_frames(nf, args.size, seed=1234)
    plant = PlantedCrowd(nf, 14, args.size, args.size, 2, num_people=args.people, seed=77, device="cpu")
    for _ in range(args.warmup):
        cpu_reference_step(cfg, arch, sd, frames, plant)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_reference_step(cfg, arch, sd, frames, plant)
    dt = time.perf_counter() - t0
    fps = nf * args.steps / dt
    cores = torch.get_num_threads()
    sample = "%d frames/step x %d steps of the same workload (fp32 CPU eager, all host threads)" % (nf, args.steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------ roofline (dominant kernels)
def _time_kernel(fn, device, iters=13, skip=3):
    """CUDA-event timing of one launch on the current stream, L2 flushed (256 MB write) between iterations."""
    import torch
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)
    times = []
    for i in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if i >= skip:
            times.append(e0.elapsed_time(e1) * 1e-3)
    return sum(times) / len(times)


def time_dw7_kernel(n, c, hw, device):
    """Stand-alone 7x7 depthwise (+bias+ReLU6, stride 1) at the stage-0 shape of the workload."""
    import torch
    from litepose_b200 import _lib
    lib = _lib.load()
    x = torch.randn((n, hw, hw, c), device=device).half()
    w = (torch.randn((49, c), device=device) * 0.1).half()
    b = torch.zeros(c, device=device)
    y = torch.empty_like(x)
    s = torch.cuda.current_stream().cuda_stream
    t = _time_kernel(lambda: _lib.check(lib.lp_dwconv_f16(x.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), n, c,
                                                          hw, hw, 7, 1, 2, s)), device)
    alg = 2 * (2 * n * c * hw * hw + 49 * c) + 4 * c
    return t, alg


def time_fused_kernel(n, ce, co, hw, device):
    """The dominant kernel of the step: fused depthwise-7x7 + projection (+identity) at the stage-0 shape."""
    import numpy as np
    import torch
    from litepose_b200 import _lib
    lib = _lib.load()
    x = (torch.rand((n, hw, hw, ce), device=device) * 3).half()
    wd = (torch.randn((49, ce), device=device) * 0.1).half()
    bd = torch.zeros(ce, device=device)
    wp = np.ascontiguousarray((np.random.RandomState(0).randn(co, ce) / ce ** 0.5).astype(np.float16)).view(np.uint16)
    wpk = np.zeros(lib.lp_pw1x1_packed_elems(ce, co), np.uint16)
    bpk = np.zeros(lib.lp_pw1x1_packed_bias_elems(co), np.float32)
    _lib.check(lib.lp_pw1x1_pack(wp.ctypes.data, None, ce, co, wpk.ctypes.data, bpk.ctypes.data))
    wpd = torch.from_numpy(wpk).view(torch.float16).to(device)
    bpd = torch.from_numpy(bpk).to(device)
    res = torch.randn((n, hw, hw, co), device=device).half()
    out = torch.empty_like(res)
    s = torch.cuda.current_stream().cuda_stream
    t = _time_kernel(lambda: _lib.check(lib.lp_dw7_project_f16(x.data_ptr(), wd.data_ptr(), bd.data_ptr(), wpd.data_ptr(),
                                                               bpd.data_ptr(), res.data_ptr(), out.data_ptr(), n, hw, hw,
                                                               ce, co, s)), device)
    # algorithmic bytes: expanded input read once, residual read, output written, weights
    alg = 2 * (n * hw * hw * ce + 2 * n * hw * hw * co + 49 * ce + ce * co) + 4 * (ce + co)
    flops = 2 * 49 * n * hw * hw * ce + 2 * n * hw * hw * ce * co
    return t, alg, flops


def time_block_kernel(n, cin, ce, co, hw, device):
    """The dominant kernel of the step: one stride-1 InvBottleneck (expand -> depthwise 7x7 -> project -> + identity) fused in
    one launch, at the stage-0 shape of the workload."""
    import numpy as np
    import torch
    from litepose_b200 import _lib
    lib = _lib.load()
    if not lib.lp_block_s1_supported(cin, ce, co):
        return None
    rs = np.random.RandomState(0)
    x = torch.randn((n, hw, hw, cin), device=device).half()
    we = np.ascontiguousarray((rs.randn(ce, cin) / cin ** 0.5).astype(np.float16)).view(np.uint16)
    wek = np.zeros(lib.lp_block_s1_wexp_elems(cin, ce), np.uint16)
    _lib.check(lib.lp_block_s1_pack_wexp(we.ctypes.data, cin, ce, wek.ctypes.data))
    wed = torch.from_numpy(wek).view(torch.float16).to(device)
    be, bd = torch.zeros(ce, device=device), torch.zeros(ce, device=device)
    wd = (torch.randn((49, ce), device=device) * 0.1).half()
    wp = np.ascontiguousarray((rs.randn(co, ce) / ce ** 0.5).astype(np.float16)).view(np.uint16)
    wpk = np.zeros(lib.lp_pw1x1_packed_elems(ce, co), np.uint16)
    bpk = np.zeros(lib.lp_pw1x1_packed_bias_elems(co), np.float32)
    _lib.check(lib.lp_pw1x1_pack(wp.ctypes.data, None, ce, co, wpk.ctypes.data, bpk.ctypes.data))
    wpd = torch.from_numpy(wpk).view(torch.float16).to(device)
    bpd = torch.from_numpy(bpk).to(device)
    out = torch.empty((n, hw, hw, co), dtype=torch.float16, device=device)
    s = torch.cuda.current_stream().cuda_stream
    t = _time_kernel(lambda: _lib.check(lib.lp_block_s1_f16(x.data_ptr(), wed.data_ptr(), be.data_ptr(), wd.data_ptr(),
                                                            bd.data_ptr(), wpd.data_ptr(), bpd.data_ptr(), 1, out.data_ptr(), n,
                                                            hw, hw, cin, ce, co, s)), device)
    # algorithmic bytes: block input read once (+ once more as the identity), block output written, weights, biases
    alg = 2 * (n * hw * hw * (2 * cin + co) + ce * cin + 49 * ce + ce * co) + 4 * (2 * ce + co)
    macs_dw = 49 * n * hw * hw * ce
    macs_tc = n * hw * hw * ce * (cin + co)
    return t, alg, macs_dw, macs_tc


def time_deconv_kernel(n, cr, cw, co, hw, device):
    """Fusion-deconv level (both ConvT branches + bias + ReLU) at the largest level of the workload."""
    import numpy as np
    import torch
    from litepose_b200 import _lib
    lib = _lib.load()
    rs = np.random.RandomState(0)
    wr = (rs.randn(cr, co, 4, 4) * 0.05).astype(np.float16).view(np.uint16)
    ww = (rs.randn(cw, co, 4, 4) * 0.05).astype(np.float16).view(np.uint16)
    wpk = np.zeros(lib.lp_deconv_packed_elems(cr, cw, co), np.uint16)
    bpk = np.zeros(lib.lp_deconv_packed_bias_elems(co), np.float32)
    _lib.check(lib.lp_deconv_pack(wr.ctypes.data, ww.ctypes.data, None, cr, cw, co, wpk.ctypes.data, bpk.ctypes.data))
    wpd = torch.from_numpy(wpk).view(torch.float16).to(device)
    bpd = torch.from_numpy(bpk).to(device)
    a = torch.randn((n, hw, hw, cr), device=device).half()
    b = torch.randn((n, hw, hw, cw), device=device).half()
    out = torch.empty((n, 2 * hw, 2 * hw, co), dtype=torch.float16, device=device)
    s = torch.cuda.current_stream().cuda_stream
    t = _time_kernel(lambda: _lib.check(lib.lp_fusion_deconv_f16(a.data_ptr(), b.data_ptr(), wpd.data_ptr(), bpd.data_ptr(),
                                                                 out.data_ptr(), n, hw, hw, cr, cw, co, s)), device)
    alg = 2 * (n * hw * hw * (cr + cw) + n * 4 * hw * hw * co + 16 * co * (cr + cw)) + 4 * co
    return t, alg


def time_forward_only(model, pipe, x_dev, device, iters=5):
    """Forward-only comparison on the same device: the hand-written engine (plain + mirrored pass, as in the step)
    against the SAME nn.Module graph executed by stock PyTorch eager ops (cuDNN fp16, cudnn.benchmark) - the op
    sequence of the reference's pose_mobilenet.py.  Informational: the stock reference itself is not on this box."""
    import copy
    import torch
    eng = pipe.engine

    def ours():
        eng.run(x_dev, flip=False, out_fp32=True, clone=False)
        eng.run(x_dev, flip=True, out_fp32=True, clone=False)

    def timed(fn, n):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / n

    t_ours = timed(ours, iters)
    old = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    try:
        eager = copy.deepcopy(model).half().eval()
        xh = x_dev.half()

        def stock():
            with torch.no_grad():
                o = eager._forward_modules(xh)
                f = eager._forward_modules(torch.flip(xh, [3]))
                return [t.float() for t in o + f]

        t_eager = timed(stock, iters)
        del eager
    finally:
        torch.backends.cudnn.benchmark = old
    torch.cuda.empty_cache()
    return t_ours, t_eager


def time_eager_gpu_e2e(args, cfg, model, device, nframes=8, warm=2):
    """The reference's own GPU path, end to end, as valid.py:195-229 runs it (SURVEY.md 8(d) "PyTorch-eager GPU"
    baseline, the denominator of the >=4x target): per image (batch 1) pinned H2D, the fp16 eager network
    (network_to_half, lib/fp16_utils/fp16util.py:87-91: half convolutions, fp32 BatchNorm; cudnn.benchmark as in
    mobile.yaml:8) on the image and on its mirror, the torch glue of lib/core/inference.py:75-208 (F.interpolate
    bilinear x2, flip-back + joint permutation, PROJECT2IMAGE, flip average), the benchmark's planted persons, then
    HeatmapParser.parse per image on the projected maps (lib/core/group.py:269-291: numpy / torch-CPU algorithm; the
    reference checkout cannot travel to this box, so its restatement oracle/group_ref runs here - baseline arm only).
    Same nn.Module graph and weights as the measured path; none of this repo's kernels are involved."""
    import copy
    import numpy as np
    import torch
    import torch.nn.functional as F
    from litepose_b200 import synth
    from litepose_b200.config import flip_index_for
    from litepose_b200.pipeline import PlantedCrowd
    from oracle import group_ref

    def bn_float(mod):
        if isinstance(mod, torch.nn.modules.batchnorm._BatchNorm):
            mod.float()
        for c in mod.children():
            bn_float(c)
        return mod

    S, J = args.size, 14
    old = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    eager = bn_float(copy.deepcopy(model).half()).eval()
    fidx = torch.tensor(flip_index_for(cfg), device=device)
    frames = synth.make_frames(nframes, S, seed=4321).pin_memory()
    plants = [PlantedCrowd(1, J, S, S, 2, num_people=args.people, seed=500 + i, device=device) for i in range(nframes)]
    parser = group_ref.HeatmapParser(cfg)
    up = lambda t, size: F.interpolate(t, size=size, mode="bilinear", align_corners=False)
    split = {"forward_glue_ms": 0.0, "parser_ms": 0.0}

    def one(i, record):
        t0 = time.perf_counter()
        with torch.no_grad():
            img = frames[i:i + 1].to(device, non_blocking=True)
            hms, tgs = [], []
            for flipped in (False, True):
                x = torch.flip(img, [3]) if flipped else img
                o0, o1 = [t.float() for t in eager._forward_modules(x.half())]
                o0 = up(o0, (o1.shape[2], o1.shape[3]))
                if flipped:
                    o0, o1 = torch.flip(o0, [3]), torch.flip(o1, [3])
                hm = (o0[:, :J] + o1[:, :J]) / 2.0
                tg = o0[:, J:]
                if flipped:
                    hm, tg = hm[:, fidx], tg[:, fidx]
                hms.append(up(hm, (S, S)))
                tgs.append(up(tg, (S, S)))
            det = ((hms[0] + hms[1]) / 2.0).contiguous()
            tag = torch.cat([t.unsqueeze(4) for t in tgs], dim=4).contiguous()
            plants[i].apply(det, tag)
            dn, tn = det.cpu().numpy(), tag.cpu().numpy()        # the reference parser works on host arrays
        t1 = time.perf_counter()
        ans, _ = parser.parse(dn, tn, True, True)
        t2 = time.perf_counter()
        if record:
            split["forward_glue_ms"] += (t1 - t0) * 1e3
            split["parser_ms"] += (t2 - t1) * 1e3
        return len(ans[0]) if len(ans) else 0

    try:
        for i in range(warm):
            one(i, False)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        found = [one(i, True) for i in range(nframes)]
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        torch.backends.cudnn.benchmark = old
        del eager
        torch.cuda.empty_cache()
    return {"frames_per_s": nframes / dt, "ms_per_frame": dt / nframes * 1e3,
            "forward_glue_ms_per_frame": split["forward_glue_ms"] / nframes,
            "parser_ms_per_frame": split["parser_ms"] / nframes, "frames": nframes, "persons_found": found[:8],
            "what": "reference flow of valid.py:195-229 on this GPU, batch 1 per image: fp16 eager nn.Module graph "
                    "(cuDNN, benchmark mode) x2 + torch glue + host HeatmapParser.parse (oracle restatement of "
                    "lib/core/group.py); wall clock incl. H2D/D2H, host threads = torch default"}


def time_variants(args, model, x_dev, plant, device, iters=5):
    """(a) the reference's nano-demo settings on the same frames: FLIP_TEST / ADJUST / REFINE off (nano_demo/core/__init__.py
    :106-116), full parser; (b) the fast_utils parser (find_peaks + KM assign, nano_demo/fast_utils/group.py:38-47) on the
    projected maps of the step: GPU plugin (whole batch) vs the C restatement of the reference's native code on one host
    core (per frame; the reference's own loop is per frame)."""
    import time as _t
    import numpy as np
    import torch
    from litepose_b200.config import get_cfg
    from litepose_b200.fast_utils.group import HeatmapParser as FastParser
    from litepose_b200.pipeline import LitePosePipeline, PlantedCrowd
    B, S = x_dev.shape[0], args.size

    def timed(fn, n):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / n

    out = {}
    cfg_fast = get_cfg(input_size=S, flip_test=False, adjust=False, refine=False)
    pipe_fast = LitePosePipeline(model, cfg_fast, use_graphs=True)
    plant1 = PlantedCrowd(B, 14, S, S, 1, num_people=args.people, seed=77, device=device)
    t = timed(lambda: pipe_fast.step_device(x_dev, plant1), iters)
    out["nano_demo_settings"] = {"frames_per_s": B / t, "ms_per_step": t * 1e3,
                                 "what": "FLIP_TEST/ADJUST/REFINE off, otherwise the bench workload (device resident)"}
    # fast_utils parser on the projected maps of that step
    st = pipe_fast._get_state(B, S, S, x_dev.dtype, plant1)
    det, tag = st["det"].clone(), st["tag"].clone()
    fp = FastParser(cfg_fast)
    tg = timed(lambda: fp.parse_batch(det, tag), iters)
    num, _ = fp.parse_batch(det, tag)
    fast = {"gpu_frames_per_s": B / tg, "gpu_ms_per_batch": tg * 1e3, "persons_found": num[:8].tolist(),
            "what": "find_peaks + KM assign on %d projected maps %dx%dx%dx%d" % (B, B, 14, S, S)}
    try:
        from oracle import fast_utils_ref as fu
        d, tm = det[:2].cpu().numpy(), tag[:2, :, :, :, 0].cpu().numpy()
        params = dict(detection_threshold=fp.params.detection_threshold, window_size=fp.params.window_size,
                      max_num_people=fp.params.max_num_people, tag_threshold=fp.params.tag_threshold,
                      joint_order=[j for j in fp.params.joint_order if j < 14][:14])
        fu.parse(d, tm, params, "port")
        t0 = _t.perf_counter()
        fu.parse(d, tm, params, "port")
        dt = _t.perf_counter() - t0
        fast["cpu_port_frames_per_s"] = 2 / dt
        fast["cpu_port_cores"] = 1
    except Exception as e:
        fast["cpu_port_error"] = str(e)[:120]
    out["fast_utils_parser"] = fast
    # (c) the whole valid.py loop body on the device (8(f) row 3): uint8 camera-order images in pinned host memory ->
    # H2D -> warpAffine + ToTensor + Normalize -> the bench step -> get_final_preds -> packed keypoints on the host
    try:
        from litepose_b200.lib.utils import transforms as T
        pipe_full = LitePosePipeline(model, get_cfg(input_size=S), use_graphs=True)
        rs = np.random.RandomState(5)
        imgs = torch.from_numpy(rs.randint(0, 256, (B, S, S, 3)).astype(np.uint8)).pin_memory()
        _, center, scale = T.get_multi_scale_size(np.empty((S, S, 3), np.uint8), S, 1.0, 1.0)
        pipe_full.set_final_preds([center] * B, [scale] * B)
        mean, std = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
        host = None

        def full():
            nonlocal host
            d = imgs.to(device, non_blocking=True)
            x, _, _ = T.resize_align_normalize_device(d, S, 1.0, 1.0, mean, std, half=True)
            packed = pipe_full.step_device(x, plant)
            if host is None:
                host = torch.empty(packed.shape, dtype=packed.dtype).pin_memory()
            host.copy_(packed, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        tf = timed(full, iters)
        out["from_uint8_images"] = {"frames_per_s": B / tf, "ms_per_step": tf * 1e3,
                                    "what": "uint8 HWC frames (pinned host) -> device warpAffine+ToTensor+Normalize -> bench "
                                            "step -> get_final_preds on the device -> keypoints on the host, synchronous"}
        del pipe_full
    except Exception as e:
        out["from_uint8_images"] = {"error": str(e)[:200]}
    # (d) multi-scale test (TEST.SCALE_FACTOR [0.5, 1, 2], valid.py:198-229): three network resolutions per frame, one
    # accumulating glue launch per scale, the parser on the summed maps; batch 8 (the 2x scale is 1024^2)
    try:
        from litepose_b200 import synth
        cfg_ms = get_cfg(input_size=S)
        cfg_ms.TEST.SCALE_FACTOR = [0.5, 1, 2]
        pipe_ms = LitePosePipeline(model, cfg_ms, use_graphs=True)
        nb = min(B, 8)
        xs = {s: synth.make_frames(nb, int(S * s), seed=31).half().to(device) for s in (0.5, 1.0, 2.0)}
        plant_ms = PlantedCrowd(nb, 14, S, S, 2, num_people=args.people, seed=78, device=device)
        tm = timed(lambda: pipe_ms.step_device_multiscale(xs, plant_ms), iters)
        out["multiscale_test"] = {"frames_per_s": nb / tm, "ms_per_step": tm * 1e3, "batch": nb, "scales": [2, 1, 0.5],
                                  "what": "TEST.SCALE_FACTOR [0.5,1,2] at base %dx%d: 6 network passes (%d^2, %d^2, %d^2) + 3 "
                                          "accumulating glue launches + parser per frame, device resident, eager launches"
                                          % (S, S, 2 * S, S, S // 2)}
        del pipe_ms, xs
    except Exception as e:
        out["multiscale_test"] = {"error": str(e)[:200]}
    del pipe_fast
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------ main arm
def main():
    args = parse_args()
    claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    import torch
    import torch.distributed as dist
    from litepose_b200 import _lib, synth
    from litepose_b200.config import get_arch, get_cfg
    from litepose_b200.lib.models.pose_mobilenet import get_pose_net
    from litepose_b200.pipeline import LitePosePipeline, PlantedCrowd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL's version / debug lines go to stdout by default: keep stdout for the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    _lib.check(lib.lp_device_check(), "lp_device_check")

    cfg = get_cfg(input_size=args.size)
    arch = get_arch(args.arch)
    torch.manual_seed(0)
    model = synth.scale_heads_(synth.randomize_bn_(get_pose_net(cfg, False, arch), 1)).eval().to(dev)
    # packed payload: 64 persons per image for the 5-person workload; crowd workloads (BASELINE config 5) carry the
    # parser's full capacity (J*K = 420 persons) so that no person can be dropped by the gather either
    pipe = LitePosePipeline(model, cfg, use_graphs=not args.no_graphs, keep=64 if args.people <= 12 else 420)
    B, S = args.batch, args.size
    frames = synth.make_frames(B, S, seed=1234, rank=rank).half().pin_memory()
    plant = PlantedCrowd(B, 14, S, S, 2, num_people=args.people, seed=77 + rank, device=dev)
    x_dev = frames.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # launches per step (non-graph single step)
    pipe.use_graphs = False
    pipe.step_device(x_dev, plant)
    torch.cuda.synchronize()
    lib.lp_reset_launch_count()
    pipe.step_device(x_dev, plant)
    torch.cuda.synchronize()
    launches_per_step = int(lib.lp_launch_count())
    pipe.use_graphs = not args.no_graphs

    # ---- device-resident throughput
    # steady-state throughput form of the step: the parser of step i (a chain of short latency-bound kernels) runs on a
    # second stream under the network passes of step i+1; every step's parser is inside the timed region (the closing
    # event is recorded after the launching stream has joined the parser stream)
    step = pipe.step_device_overlapped if not args.no_graphs else (lambda a, b: (pipe.step_device(a, b), None))
    for _ in range(max(args.warmup, 3)):
        step(x_dev, plant)
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        packed, parsed = step(x_dev, plant)
    if parsed is not None:
        torch.cuda.current_stream().wait_event(parsed)
    e1.record()
    barrier()
    # the payload buffers are reused by the steps below: keep the last timed step's result now
    last_packed = packed.cpu().numpy() if args.dump_outputs else None
    t_dev = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / t_dev

    # ---- end to end through the public asynchronous API (LitePosePipeline.submit / collect): pinned host frames in,
    # keypoints of every rank on rank 0's host out.  Two steps are in flight: the H2D copy of step i+1 and the NCCL gather
    # + D2H copy of step i-1 overlap the compute of step i; the host consumes the keypoints of step i-1 while step i runs
    # (no per-step device synchronisation).  Every step's result is waited for inside the timed region.
    group = dist.group.WORLD if world > 1 else None
    packed0 = pipe.step_device(x_dev, plant)
    h2d_bytes = frames.numel() * frames.element_size()
    d2h_bytes = packed0.numel() * packed0.element_size() * world
    last_host = [None]

    def e2e_steps(k):
        prev = None
        for i in range(k):
            t = pipe.submit(frames, plant, group=group, dst=0)
            if prev is not None:
                h = pipe.collect(prev, unpack=False)
                if h is not None:
                    last_host[0] = h
            prev = t
        h = pipe.collect(prev, unpack=False)
        if h is not None:
            last_host[0] = h

    e2e_steps(max(args.warmup, 3))
    barrier()
    t0 = time.perf_counter()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    e2e_steps(args.steps)          # returns after the LAST step's keypoints are on the host
    c1.record()
    barrier()
    t_wall = max_over_ranks(time.perf_counter() - t0)     # host wall clock: submit of step 0 -> last keypoints on the host
    t_e2e = max_over_ranks(max(c0.elapsed_time(c1) * 1e-3, 0.0))
    # the result stream is not the launching stream: the device events on the launching stream end before the last D2H
    # copy, so the e2e number is the LARGER of the two clocks
    t_e2e = max(t_e2e, t_wall)
    e2e_value = world * B * args.steps / t_e2e
    host_out = last_host[0]
    if args.dump_outputs and rank == 0:
        # packed: [N, keep*J*(3+T) + keep + 1] of rank 0 (keypoints, scores, person count; LitePosePipeline.unpack);
        # e2e_packed: [ranks, N, ...] as collect() hands it to rank 0's host
        dump_outputs(args.dump_outputs, {"packed": payload_as_received(last_packed, pipe.keep),
                                         "e2e_packed": payload_as_received(host_out.numpy(), pipe.keep)})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # sanity: the planted persons are found
    found = [int(v) for v in host_out[0][:, -1].tolist()]

    # ---- roofline of the dominant kernel (dw7x7 stage-0 shape of this workload)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    c0 = arch["backbone_setting"][0]["channel"]
    c_stage0 = 6 * c0
    t_f, alg_f, flops_f = time_fused_kernel(B, c_stage0, c0, S // 4, dev)
    t_k, alg = time_dw7_kernel(B, c_stage0, S // 4, dev)
    blk = time_block_kernel(B, c0, c_stage0, c0, S // 4, dev)
    src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    # CUDA-core multiply-add ceiling of this part, measured by tools/microbench/fma_rates.cu (profiles/r2_fma_rates.jsonl):
    # HFMA2 = 126 MAC/clk/SM (FFMA 93, FHFMA 108) -> x SMs x the clock sampled during the step
    try:
        with open(os.path.join(ROOT, "profiles", "r2_fma_rates.jsonl")) as f:
            rates = [json.loads(l) for l in f if l.strip()]
        hfma2_mac_clk_sm = max(r["macs_per_clk_per_sm"] for r in rates if "macs_per_clk_per_sm" in r)
    except Exception:
        hfma2_mac_clk_sm = 126.0
    sm_mhz = (clocks or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    fma_peak_tmacs = hfma2_mac_clk_sm * n_sm * sm_mhz * 1e6 / 1e12
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")) as f:
            tj = json.load(f)
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
    except Exception:
        pass
    fused_entry = {"kernel": "dw_project_kernel<7,0> (depthwise7x7+projection+identity on the HBM-resident expanded tensor) "
                             "%dx%dx%dx%d->%d" % (B, S // 4, S // 4, c_stage0, c0),
                   "achieved": alg_f / t_f / 1e9, "frac": alg_f / t_f / 1e9 / peak_gbs, "algorithmic_bytes": alg_f,
                   "avg_launch_us": t_f * 1e6, "dw_tmacs": (flops_f / 2) / t_f / 1e12,
                   "fma_frac": 49 * B * (S // 4) ** 2 * c_stage0 / t_f / 1e12 / fma_peak_tmacs}
    if blk is not None:
        t_b, alg_b, macs_dw, macs_tc = blk
        achieved = alg_b / t_b / 1e9
        roofline = {"bound": "hbm",
                    "kernel": "block_s1_kernel (one stride-1 InvBottleneck: expand on tcgen05 -> depthwise7x7 -> projection "
                              "-> identity, the 6x tensor stays on chip) %dx%dx%dx%d->%d->%d" % (B, S // 4, S // 4, c0, c_stage0, c0),
                    "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                    "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": alg_b,
                    "avg_launch_us": t_b * 1e6, "peak_source": src,
                    "limiter": "CUDA-core fp16 FMA pipe (49 MAC per expanded element; HBM carries only the narrow block "
                               "input/output after block fusion, so the HBM fraction is low by construction)",
                    "fma_pipe": {"achieved_tmacs": macs_dw / t_b / 1e12, "peak_tmacs": fma_peak_tmacs,
                                 "frac": macs_dw / t_b / 1e12 / fma_peak_tmacs, "peak_mac_per_clk_per_sm": hfma2_mac_clk_sm,
                                 "sm_mhz": sm_mhz, "peak_source": "profiles/r2_fma_rates.jsonl (HFMA2, measured on this pool)"},
                    "tensor_tflops": 2 * macs_tc * 1.89 / t_b / 1e12,
                    "unfused_dw_project_kernel": fused_entry,
                    "unfused_dwconv_kernel": {"kernel": "dwconv_kernel<7,1> %dx%dx%dx%d" % (B, S // 4, S // 4, c_stage0),
                                              "achieved": alg / t_k / 1e9, "frac": alg / t_k / 1e9 / peak_gbs,
                                              "algorithmic_bytes": alg, "avg_launch_us": t_k * 1e6}}
    else:
        roofline = dict(fused_entry)
        roofline.update({"bound": "hbm", "peak": peak_gbs, "unit": "GB/s", "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": src})

    ds = arch["deconv_setting"]
    cr_l2, cw_l2 = ds[-2], arch["backbone_setting"][0]["channel"]
    try:
        t_d, alg_d = time_deconv_kernel(B, cr_l2, cw_l2, ds[-1], S // 4, dev)
        roofline["fusion_deconv_kernel"] = {
            "kernel": "fusion deconv level %d: %dx%dx%dx(%d+%d)->%d" % (len(ds) - 1, B, S // 4, S // 4, cr_l2, cw_l2, ds[-1]),
            "achieved": alg_d / t_d / 1e9, "frac": alg_d / t_d / 1e9 / peak_gbs, "algorithmic_bytes": alg_d,
            "avg_launch_us": t_d * 1e6}
    except Exception as e:   # never lose the bench line over the auxiliary entry
        roofline["fusion_deconv_kernel"] = {"error": str(e)[:200]}

    fwd = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            t_ours, t_eager = time_forward_only(model, pipe, x_dev, dev)
            fwd = {"ours_fps": B / t_ours, "torch_eager_fp16_fps": B / t_eager, "ratio": t_eager / t_ours,
                   "what": "forward only, plain + mirrored pass per frame, batch %d; torch_eager = the same nn.Module "
                           "graph on stock PyTorch ops (cuDNN fp16, benchmark mode), not the reference checkout" % B}
        except Exception as e:
            fwd = {"error": str(e)[:200]}

    # ---- the reference's own GPU path end to end (8(d): denominator of the >=4x target), N=1 only
    eager_e2e = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            eager_e2e = time_eager_gpu_e2e(args, cfg, model, dev)
            eager_e2e["e2e_ratio"] = e2e_value / eager_e2e["frames_per_s"]
        except Exception as e:
            eager_e2e = {"error": str(e)[:200]}

    # ---- secondary variants (N=1 only, short): the nano-demo "fast" settings and the fast_utils parser (8(d), 8(f) row 2)
    variants = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            variants = time_variants(args, model, x_dev, plant, dev)
        except Exception as e:
            variants = {"error": str(e)[:200]}

    # ---- CPU baseline (oracle port) on a bounded sample
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        ccfg, carch, sd = cpu_reference_setup(args)
        nf = 2
        fr = synth.make_frames(nf, S, seed=1234)
        cp = PlantedCrowd(nf, 14, S, S, 2, num_people=args.people, seed=77, device="cpu")
        cpu_reference_step(ccfg, carch, sd, fr, cp)          # warm-up
        reps = max(1, args.cpu_sample // nf)
        t0 = time.perf_counter()
        for _ in range(reps):
            cpu_reference_step(ccfg, carch, sd, fr, cp)
        dt = time.perf_counter() - t0
        cpu = {"value": nf * reps / dt, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": "%d frames of the same workload (oracle port: fp32 eager CPU forward x2 + glue + parser)"
                         % (nf * reps)}

    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes * world,
                "d2h_bytes_per_step": d2h_bytes, "ms_per_step": t_e2e / args.steps * 1e3,
                "wall_ms_per_step": t_wall / args.steps * 1e3},
        "gpu_launches": launches_per_step * args.steps * 2 * world,
        "launches_per_step": launches_per_step,
        "cuda_graphs": not args.no_graphs,
        "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "forward_only": fwd, "eager_gpu_e2e": eager_e2e,
        "variants": variants,
        "persons_found_rank0": found[:8],
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
