#!/usr/bin/env python
"""bench.py -- training images/sec of the BTS hot path on B200 (BASELINE.json metric), one JSON line.

    python bench.py --gpus N --steps K --warmup W [--config K16|N4|R8|T1|LPG]    # our arm (torchrun launches N>1)
    python bench.py --impl reference --gpus N --steps K ...                      # reference arm: the reference on host cores
    python bench.py ... --dump-outputs DIR     # also write what the last timed step computed to DIR/<name>.npy

Default workload K16 (BASELINE.json configs[1], the config the metric is quoted on): DenseNet-161 encoder, 352x704
synthetic RGB->depth, batch 16 PER GPU (weak scaling), train mode (batch-stat BN), silog loss (lambda .85), backward,
AdamW step with the two parameter groups and poly LR of bts_main.py:371-373,456-460.  A "step" = zero_grad + forward +
loss + backward + optimizer step over one batch.  Other configs (BASELINE.json configs[0,2,3,4]) via --config:
N4 = DN-161 416x544 NYU-shape B=4/GPU, R8 = ResNeXt-101 352x704 B=8/GPU, T1 = DN-121 416x544 B=1 eval forward,
LPG = the LPG-only microbench (r = 8/4/2, H=W = 256..1024, HBM regime and B=16 regime).

Keys (see DESIGN.md section 5):
  value          K timed steps, inputs resident in HBM, CUDA events on the launching stream, max over ranks
  e2e            same metric with the batch starting in pinned host memory (H2D inside the timed region) and the loss read
                 back (D2H) every step
  roofline       the DOMINANT kernel of the step (conv_tc_kernel: every conv forward and dgrad): nominal FLOPs of all of
                 its launches in one step / the sum of their CUDA-event durations inside a real step (FLOP-weighted), against
                 the parity-mode tensor roof = measured TF32 GEMM peak (sustained: the kernel is timed inside a long step) / 3
  roofline_wgrad same for the wgrad kernels;  roofline_lpg: the LPG fwd+bwd pair against the measured HBM peak (burst:
                 timed in isolation);  roofline_step: whole step, nominal conv FLOPs / step time
  peaks_live     TF32 GEMM peak measured by this run the way MEASURED_PEAKS.json was made for bf16 (cuBLAS 8192^3)
  gpu_baseline   the reference model (unmodified pytorch/bts.py when oracle/_ref travelled, else the oracle port) under
                 stock torch-eager + cuDNN on the same GPU, fp32 (TF32 off) and with PyTorch's default cudnn TF32
  cpu_baseline   the reference on the box's host cores (bounded sample)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# name: encoder, H, W, batch per GPU, dataset, max_depth, focal, valid fraction of gt, mask threshold, train,
#       nominal conv GFLOP per image (BASELINE.md section 3: train = fwd+dgrad+wgrad; T1 = forward only)
CONFIGS = {
    "K16": dict(encoder="densenet161_bts", H=352, W=704, B=16, dataset="kitti", max_depth=80.0, focal=721.5377,
                valid=0.2, thr=1.0, train=True, gflop=588.0,
                workload="K16: DenseNet-161 encoder, 352x704 KITTI-shape synthetic, batch 16/GPU, train step "
                         "(fwd + silog + bwd + AdamW), random-init weights",
                metric="training images/sec (352x704, DenseNet-161)"),
    "N4": dict(encoder="densenet161_bts", H=416, W=544, B=4, dataset="nyu", max_depth=10.0, focal=518.8579,
               valid=0.95, thr=0.1, train=True, gflop=537.0,
               workload="N4: DenseNet-161 encoder, 416x544 NYU-shape synthetic, batch 4/GPU, train step "
                        "(fwd + silog + bwd + AdamW), random-init weights",
               metric="training images/sec (416x544, DenseNet-161)"),
    "R8": dict(encoder="resnext101_bts", H=352, W=704, B=8, dataset="kitti", max_depth=80.0, focal=721.5377,
               valid=0.2, thr=1.0, train=True, gflop=893.0,
               workload="R8: ResNeXt-101 (32x8d) encoder, 352x704 KITTI-shape synthetic, batch 8/GPU, train step "
                        "(fwd + silog + bwd + AdamW), random-init weights",
               metric="training images/sec (352x704, ResNeXt-101)"),
    "T1": dict(encoder="densenet121_bts", H=416, W=544, B=1, dataset="nyu", max_depth=10.0, focal=518.8579,
               valid=0.95, thr=0.1, train=False, gflop=119.5,
               workload="T1: DenseNet-121 encoder, single 416x544 frame, eval-mode forward only (bts_test.py shape), "
                        "random-init weights",
               metric="inference images/sec (416x544, DenseNet-121, batch 1)"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "fallback (B200_PROFILING.md)"}


def synth_batch(cfg, B, seed, dev="cpu", pin=False):
    """SURVEY 8d synthetic inputs: image randn, focal (float64 like the DataLoader collate), depth U(0,max_depth) with a
    Bernoulli validity mask (KITTI-like sparse 20 % / NYU-like dense 95 %, else 0)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    H, W = cfg["H"], cfg["W"]
    img = torch.randn(B, 3, H, W, generator=g)
    gt = torch.rand(B, 1, H, W, generator=g) * cfg["max_depth"]
    gt = torch.where(torch.rand(B, 1, H, W, generator=g) < cfg["valid"], gt, torch.zeros_like(gt))
    focal = torch.full((B,), cfg["focal"], dtype=torch.float64)
    if pin:
        return img.pin_memory(), focal.pin_memory(), gt.pin_memory()
    return img.to(dev), focal.to(dev), gt.to(dev)


def make_optimizer(model, torch, fused=False):
    """bts_main.py:371-373 (lr 1e-4, eps 1e-3, wd 1e-2 encoder / 0 decoder: arguments_train_eigen.txt).
    fused: bts_b200.optim.FusedAdamW -- the same optimizer (state_dict-compatible, ulp-level parity test) as one kernel."""
    m = model.module if hasattr(model, "module") else model
    groups = [{"params": m.encoder.parameters(), "weight_decay": 1e-2}, {"params": m.decoder.parameters(), "weight_decay": 0}]
    if fused:
        from bts_b200.optim import FusedAdamW
        return FusedAdamW(groups, lr=1e-4, eps=1e-3)
    return torch.optim.AdamW(groups, lr=1e-4, eps=1e-3)


def freeze_like_set_misc(model):
    """bts_main.py:217-247 default ('Fixing first conv layer'): parameters whose name contains one of
    ['base_model.conv1', '.bn'] (ResNet family) / ['conv0', 'norm'] (DenseNet) are frozen."""
    names = [n for n, _ in model.encoder.named_parameters()]
    dense = any("denseblock" in n for n in names)
    keys = ("conv0", "norm") if dense else ("base_model.conv1", ".bn")
    for name, p in model.encoder.named_parameters():
        if any(x in name for x in keys):
            p.requires_grad = False


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.p, self.start = [], None, 0
        try:
            self.p = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append(line.strip())

    def mark(self):
        """the timed region starts now: earlier samples are dropped"""
        self.start = len(self.rows)

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[self.start:]:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def usable_cores():
    """host cores this process may actually use: affinity mask, capped by the cgroup CPU quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


# ------------------------------------------------------------------------------------------------ reference legs
def _reference_model(cfg, torch):
    """(model, silog criterion, kind, description): the UNMODIFIED reference pytorch/bts.py when it is reachable
    (oracle/_ref/bts.py, copied there by `make -C oracle`, travels with the working tree; /root/reference in the build
    container), else the oracle port.  Test/bench infrastructure only."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_shim
    p = types.SimpleNamespace(encoder=cfg["encoder"], max_depth=cfg["max_depth"], dataset=cfg["dataset"], bts_size=512)
    torch.manual_seed(0)
    if ref_shim.reference_available():
        R = ref_shim.load_reference()
        m = R.BtsModel(p)
        m.decoder.apply(R.weights_init_xavier)
        crit = R.silog_loss(variance_focus=0.85)
        return m, (lambda est, gt, mask: crit.forward(est, gt, mask)), "reference", "unmodified pytorch/bts.py (%s)" % ref_shim.REFERENCE_DIR
    import bts_oracle as O
    m = O.OracleModel(cfg["encoder"], cfg["max_depth"], cfg["dataset"], 512)
    return m, (lambda est, gt, mask: O.silog(est, gt, mask, 0.85)), "port", "oracle/bts_oracle.py OracleModel"


def cpu_reference_steps(cfg, steps, warmup, B=2, budget_s=None):
    """The reference on all host cores: one train step (or eval forward for T1) per sample batch of B images.
    budget_s: stop timing after this many seconds (bounded sample), else run every step."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_shim
    cores = usable_cores()
    torch.set_num_threads(cores)
    with ref_shim.cuda_is_identity():          # the reference's LPG calls .cuda() inside forward (bts.py:140,143)
        m, crit, kind, what = _reference_model(cfg, torch)
        train = cfg["train"]
        if not train:
            B = 1
        m.train() if train else m.eval()
        opt = make_optimizer(m, torch) if train else None
        img, focal, gt = synth_batch(cfg, B, 1)
        times = []
        t_start = time.perf_counter()
        for i in range(warmup + steps):
            if budget_s is not None and times and time.perf_counter() - t_start > budget_s:
                break                                  # bounded sample: keep the bench within minutes on slow hosts
            t0 = time.perf_counter()
            if train:
                opt.zero_grad()
                out = m(img, focal)
                loss = crit(out[4], gt, gt > cfg["thr"])
                loss.backward()
                opt.step()
                float(loss.detach())
            else:
                with torch.no_grad():
                    out = m(img, focal)
                float(out[4].sum())
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    total = sum(times)
    return {"value": B * len(times) / total, "unit": "images/s", "cores": cores, "kind": kind,
            "sample": "%s, torch CPU fp32, %d threads, %s %dx%d, B=%d %s, %d timed steps after %d warm-up"
                      % (what, cores, cfg["encoder"], cfg["H"], cfg["W"], B,
                         "train step (fwd+silog+bwd+AdamW)" if train else "eval forward", len(times), warmup),
            "ms_per_step": 1e3 * total / len(times)}


def gpu_reference_steps(cfg, torch, dev, steps=5, warmup=3):
    """SURVEY 8d / BASELINE.md section 4 'second baseline (the bar to beat)': the reference model under stock torch-eager +
    cuDNN on the same GPU -- fp32 with TF32 disabled (the parity-grade comparison) and with PyTorch's default
    cudnn.allow_tf32=True (what a user gets out of the box), cudnn.benchmark=True as bts_main.py:402."""
    out = {}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    m, crit, kind, what = _reference_model(cfg, torch)
    train = cfg["train"]
    m.to(dev)
    m.train() if train else m.eval()
    opt = make_optimizer(m, torch) if train else None
    B = cfg["B"]
    img, focal, gt = synth_batch(cfg, B, 1, dev)
    st = torch.cuda.current_stream()

    def step():
        if train:
            opt.zero_grad()
            o = m(img, focal)
            loss = crit(o[4], gt, gt > cfg["thr"])
            loss.backward()
            opt.step()
        else:
            with torch.no_grad():
                m(img, focal)

    try:
        for label, tf32 in (("fp32", False), ("tf32_default", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            for _ in range(warmup):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(steps):
                step()
            e1.record(st)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[label] = {"value": B / (ms / 1e3), "unit": "images/s", "ms_per_step": ms}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = saved
    out["kind"] = kind
    out["what"] = ("%s on cuda, torch-eager + cuDNN, cudnn.benchmark=True, %s %dx%d B=%d %s, %d timed steps after %d warm-up; "
                   "fp32 = cudnn.allow_tf32 False (parity-grade), tf32_default = PyTorch's default cudnn.allow_tf32 True"
                   % (what, cfg["encoder"], cfg["H"], cfg["W"], B, "train step" if train else "eval forward", steps, warmup))
    del m, opt
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ live peaks
def tf32_peak(torch, secs=3.0, n=8192):
    """TF32 dense GEMM peak, measured like MEASURED_PEAKS.json's bf16 figures (torch.matmul -> cuBLAS, 8192^3):
    best of 10 = burst (for a kernel timed alone), back to back for `secs` s = sustained (for a kernel timed in a step)."""
    saved = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(n, n, device="cuda")
        b = torch.randn(n, n, device="cuda")
        c = torch.empty(n, n, device="cuda")
        fl = 2.0 * n ** 3
        for _ in range(3):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0, k = time.time(), 0
        e0.record()
        while time.time() - t0 < secs:
            for _ in range(20):
                torch.matmul(a, b, out=c)
            k += 20
            torch.cuda.synchronize()
        e1.record()
        torch.cuda.synchronize()
        sus = e0.elapsed_time(e1) / k
    finally:
        torch.backends.cuda.matmul.allow_tf32 = saved
    del a, b, c
    torch.cuda.empty_cache()
    return {"tf32_tflops": fl / best / 1e9, "tf32_tflops_sustained": fl / sus / 1e9,
            "how": "torch.matmul fp32, allow_tf32 (cuBLAS TF32) %d^3: best of 10 (burst); back to back %.0f s (sustained)" % (n, secs)}


# ------------------------------------------------------------------------------------------------ LPG microbench
def _lpg_planes(torch, dev, Bn, h, w, r, max_depth):
    import math
    g = torch.Generator(device=dev).manual_seed(r)
    z = torch.randn(Bn, 3, h, w, device=dev, generator=g)
    th = torch.sigmoid(z[:, 0]) * math.pi / 3
    ph = torch.sigmoid(z[:, 1]) * math.pi * 2
    return torch.stack([torch.sin(th) * torch.cos(ph), torch.sin(th) * torch.sin(ph), torch.cos(th),
                        torch.sigmoid(z[:, 2]) * max_depth], 1).contiguous()


def _lpg_time(torch, dev, Bn, side, r, reps=20, flush=None):
    """average CUDA-event duration of bts_lpg_fwd / bts_lpg_bwd launched back to back through the C ABI.
    flush: a buffer > L2 rewritten between launches (B=16 regime: working set < 126 MB L2, so each launch is timed alone)."""
    import ctypes
    from bts_b200 import _lib
    L = _lib.lib()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    st = torch.cuda.current_stream()
    sp = ctypes.c_void_p(st.cuda_stream)
    h = side // r
    plane = _lpg_planes(torch, dev, Bn, h, h, r, 80.0)
    depth = torch.empty(Bn, side, side, device=dev)
    dy = torch.randn(Bn, side, side, device=dev)
    dplane = torch.empty_like(plane)
    fwd = lambda: L.bts_lpg_fwd(vp(plane), vp(depth), Bn, h, h, r, 0, sp)
    bwd = lambda: L.bts_lpg_bwd(vp(dy), vp(plane), vp(dplane), Bn, h, h, r, 0, 0, sp)
    res = []
    for fn in (fwd, bwd):
        for _ in range(3):
            assert fn() == 0
        torch.cuda.synchronize()
        if flush is None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(reps):
                fn()
            e1.record(st)
            torch.cuda.synchronize()
            res.append(e0.elapsed_time(e1) / reps)
        else:
            ts = []
            for _ in range(reps):
                flush.add_(1.0)                           # evict L2
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                fn()
                e1.record(st)
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            res.append(statistics.median(ts))
        _lib.count(reps + 3)
    px = float(Bn) * side * side
    bf, bb = 4.0 * px * (1 + 4.0 / r ** 2), 4.0 * px * (1 + 8.0 / r ** 2)
    mf, mb = res
    del plane, depth, dy, dplane
    return {"B": Bn, "side": side, "r": r, "fwd_ms": mf, "bwd_ms": mb, "fwd_gbs": bf / mf / 1e6, "bwd_gbs": bb / mb / 1e6,
            "fwd_bwd_gbs": (bf + bb) / (mf + mb) / 1e6, "algorithmic_bytes": bf + bb}


def lpg_roofline(torch, dev, pk):
    """LPG fwd+bwd r=8/4/2 at 1024^2, batch 128: the output is 512 MB (>> 126 MB L2; consecutive launches cannot hit in
    L2).  Algorithmic bytes: fwd 4*px*(1+4/r^2), bwd 4*px*(1+8/r^2)  (BASELINE.md section 3)."""
    out = {}
    for r in (8, 4, 2):
        t = _lpg_time(torch, dev, 128, 1024, r)
        out["r%d" % r] = t
    torch.cuda.empty_cache()
    a = out["r8"]["fwd_bwd_gbs"]
    return {"bound": "hbm", "kernel": "lpg_fwd_vec<8> + lpg_bwd_vec<8> (fwd+bwd, r=8, 128x1024x1024, output 512 MB >> L2, "
                                      "20 back-to-back launches each, timed in isolation -> burst peak)",
            "achieved": a, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": a / pk["hbm_gbs"], "peak_source": pk["source"],
            # dram__bytes_read.sum + dram__bytes_write.sum of one (fwd, bwd) launch pair, `ncu --set full` capture
            # profiles/r01_lpg_r8_v2.ncu-rep of this same microbench: fwd 33.6 + 479.3 MB, bwd 570.4 + 32.3 MB
            "traffic": 1115.6e6, "traffic_unit": "bytes per fwd+bwd launch pair (ncu, profiles/r01_lpg_r8_v2.ncu-rep)",
            "algorithmic_bytes": out["r8"]["algorithmic_bytes"], "sweep": out}


def run_lpg_config(args):
    """--config LPG (BASELINE.json configs[4]): r in {8,4,2} x H=W in {256,384,512,768,1024}; two regimes per point:
    'hbm' = batch sized so the output is >= 512 MB (working set >> L2), 'b16' = batch 16 with an L2 flush between launches."""
    import torch
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    from bts_b200 import _lib
    _lib.lib()
    pk = peaks()
    flush = torch.zeros(64 * 1024 * 1024, device=dev)         # 256 MB > 126 MB L2
    rows = []
    l0 = _lib.launches
    for r in (8, 4, 2):
        for side in (256, 384, 512, 768, 1024):
            Bh = max(16, (512 * 1024 * 1024 + 4 * side * side - 1) // (4 * side * side))
            a = _lpg_time(torch, dev, Bh, side, r, reps=args.steps)
            b = _lpg_time(torch, dev, 16, side, r, reps=args.steps, flush=flush)
            rows.append({"r": r, "side": side, "hbm": {k: a[k] for k in ("B", "fwd_ms", "bwd_ms", "fwd_gbs", "bwd_gbs", "fwd_bwd_gbs")},
                         "b16": {k: b[k] for k in ("B", "fwd_ms", "bwd_ms", "fwd_gbs", "bwd_gbs", "fwd_bwd_gbs")}})
            torch.cuda.empty_cache()
    vals = [x["hbm"]["fwd_bwd_gbs"] for x in rows]
    res = {"metric": "LPG fwd+bwd GB/s vs HBM peak", "value": statistics.median(vals), "unit": "GB/s", "n_gpus": 1,
           "steps": args.steps, "warmup": 3, "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": "LPG-u: plane-to-depth fwd+bwd, r=8/4/2, H=W 256..1024, 1 GPU; value = median over the 15 "
                                  "HBM-regime points", "l2": "hbm regime: outputs >= 512 MB; b16 regime: 256 MB flush write between launches"},
           "roofline": {"bound": "hbm", "achieved": statistics.median(vals), "peak": pk["hbm_gbs"], "unit": "GB/s",
                        "frac": statistics.median(vals) / pk["hbm_gbs"], "min_frac": min(vals) / pk["hbm_gbs"],
                        "peak_source": pk["source"], "traffic": None},
           "gpu_launches": _lib.launches - l0, "sweep": rows}
    return res


# ------------------------------------------------------------------------------------------------ engine self-check
# Round-2 fast paths (lean MMA issue loops, BatchNorm-backward sums in the dgrad epilogue, fused AdamW, CUDA-graph capture)
# each have a switch.  Before timing, a SUBPROCESS checks each against an independent computation on the GPU at hand and the
# bench only enables what passed -- a kernel bug then costs speed and is reported in the JSON line ("selfcheck"), it does not
# silently produce a wrong number or kill the run (a device-side trap in the child leaves this process's context intact).
SELFCHECK_FEATURES = ["lean_issue", "bn_onepass", "epi_bnbwd", "fused_adamw"]


def selfcheck_child(enabled):
    """runs in the child: prints 'CHECK <feature> <ok|fail> <detail>' lines; a crash after 'BEGIN <feature>' = that feature"""
    import torch
    import torch.nn.functional as F
    from bts_b200 import _lib, conv, fused
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    torch.backends.cudnn.allow_tf32 = False
    g = torch.Generator().manual_seed(0)

    def relerr(a, b):
        return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))

    def engine_ok():
        worst = 0.0
        for (B, Cin, H, W, Cout, k, pad, dil) in [(2, 192, 12, 20, 48, 3, 1, 1), (1, 240, 16, 24, 192, 1, 0, 1),
                                                    (1, 128, 10, 12, 256, 3, 3, 3), (2, 36, 24, 32, 32, 3, 1, 1)]:
            x = torch.randn(B, Cin, H, W, generator=g).to(dev).contiguous(memory_format=torch.channels_last).requires_grad_(True)
            w = (torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5).to(dev).requires_grad_(True)
            y = conv.conv2d(x, w, 1, pad, dil)
            gy = torch.randn(y.shape, generator=g).to(dev).contiguous(memory_format=torch.channels_last)
            y.backward(gy)
            xr, wr = x.detach().clone().requires_grad_(True), w.detach().clone().requires_grad_(True)
            yr = F.conv2d(xr, wr, None, 1, pad, dil)
            yr.backward(gy)
            torch.cuda.synchronize()
            worst = max(worst, relerr(y.detach(), yr.detach()), relerr(x.grad, xr.grad), relerr(w.grad, wr.grad))
        return worst < 2e-4, "worst rel-to-scale error %.2e vs torch fp32 conv (fwd/dgrad/wgrad, 4 layer shapes)" % worst

    print("BEGIN lean_issue", flush=True)
    L.bts_conv_set_issue_mode(1 if "lean_issue" in enabled else 0)
    ok, det = engine_ok()
    if "lean_issue" not in enabled:
        print("CHECK lean_issue fail disabled after a crash; legacy loops: %s %s" % ("ok" if ok else "FAIL", det), flush=True)
    elif not ok:
        L.bts_conv_set_issue_mode(0)
        ok2, det2 = engine_ok()
        print("CHECK lean_issue fail %s; legacy loops: %s %s" % (det, "ok" if ok2 else "FAIL", det2), flush=True)
    else:
        print("CHECK lean_issue ok %s" % det, flush=True)

    import torchvision
    blk = torchvision.models.densenet._DenseBlock(3, 64, 4, 32, 0.0).to(dev).train()
    from bts_b200 import model as M
    M.adopt_convs(torch.nn.Sequential(blk))
    xin = torch.randn(2, 64, 12, 16, generator=g).to(dev).contiguous(memory_format=torch.channels_last)

    def block_grads(epi, onepass):
        fused.EPI_BNBWD, fused.BN_ONEPASS = epi, onepass
        for q in blk.parameters():
            q.grad = None
        xi = xin.clone().requires_grad_(True)
        out = blk(xi)
        out.square().mean().backward()
        torch.cuda.synchronize()
        return [xi.grad.clone()] + [q.grad.clone() for q in blk.parameters()]

    base = block_grads(False, False)
    for feat, epi, onepass in (("bn_onepass", False, True), ("epi_bnbwd", True, False)):
        print("BEGIN %s" % feat, flush=True)
        worst = max(relerr(a, b) for a, b in zip(block_grads(epi, onepass), base))
        print("CHECK %s %s worst rel error %.2e vs the reduce + apply passes (dense block, all gradients)"
              % (feat, "ok" if worst < 1e-4 else "fail", worst), flush=True)

    print("BEGIN fused_adamw", flush=True)
    from bts_b200.optim import FusedAdamW
    pa = [torch.nn.Parameter(torch.randn(*sh, generator=g).to(dev)) for sh in [(48, 192, 3, 3), (7,), (513,), (64, 36, 3, 3)]]
    pb = [torch.nn.Parameter(q.detach().clone()) for q in pa]
    oa = torch.optim.AdamW([{"params": pa[:2], "weight_decay": 1e-2}, {"params": pa[2:], "weight_decay": 0}], lr=1e-4, eps=1e-3)
    ob = FusedAdamW([{"params": pb[:2], "weight_decay": 1e-2}, {"params": pb[2:], "weight_decay": 0}], lr=1e-4, eps=1e-3, repack=False)
    for _ in range(3):
        for a, b in zip(pa, pb):
            gr = torch.randn(a.shape, generator=g).to(dev)
            a.grad, b.grad = gr.clone(), gr.clone()
        oa.step()
        ob.step()
    torch.cuda.synchronize()
    ok = all(torch.allclose(a, b, rtol=1e-6, atol=1e-9) for a, b in zip(pa, pb))
    print("CHECK fused_adamw %s vs torch.optim.AdamW after 3 steps" % ("ok" if ok else "fail"), flush=True)


def _child_env():
    """the child sees exactly this rank's GPU as cuda:0"""
    local = int(os.environ.get("LOCAL_RANK", "0"))
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    ids = [v for v in vis.split(",") if v] if vis else None
    dev = ids[local] if ids and local < len(ids) else str(local)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=dev)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    return env


def run_selfcheck():
    """parent side: returns {feature: (bool ok, detail)}; at most len(features)+1 child runs"""
    enabled = list(SELFCHECK_FEATURES)
    results = {}
    for _attempt in range(len(SELFCHECK_FEATURES) + 1):
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--selfcheck-child", ",".join(enabled) or "none"],
                                 capture_output=True, text=True, timeout=600, cwd=ROOT, env=_child_env())
            text = out.stdout
        except subprocess.TimeoutExpired as e:
            text = (e.stdout or b"").decode() if isinstance(e.stdout, bytes) else (e.stdout or "")
        begun, crashed = None, None
        for line in text.splitlines():
            f = line.split(None, 3)
            if len(f) >= 2 and f[0] == "BEGIN":
                begun = f[1]
            elif len(f) >= 3 and f[0] == "CHECK":
                results[f[1]] = (f[2] == "ok", f[3] if len(f) > 3 else "")
                begun = None
        if begun is not None:                      # the child died inside this feature's check
            crashed = begun
            results[crashed] = (False, "child process crashed during the check")
        if crashed is None or crashed not in enabled:
            break
        enabled.remove(crashed)
    for f in SELFCHECK_FEATURES:
        results.setdefault(f, (False, "not reached"))
    return results


class StdoutToStderr:
    """While active, file descriptor 1 points at stderr: library chatter (e.g. the "NCCL version ..." banner NCCL prints on
    stdout at communicator creation) cannot precede the ONE JSON line this script owes its caller on stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def run_ours(args):
    if args.config == "LPG":
        if int(os.environ.get("RANK", "0")) == 0:       # single-GPU microbench (BASELINE.json configs[4]: "1 GPU")
            with StdoutToStderr():
                res = run_lpg_config(args)
            print(json.dumps(res), flush=True)
        return
    with StdoutToStderr():
        res, rank, dist = _run_ours(args)
    if rank == 0:
        print(json.dumps(res), flush=True)
    if dist is not None:
        with StdoutToStderr():
            dist.destroy_process_group()


def conv_rooflines(torch, conv, step_fn, pk_tf32):
    """One extra, untimed training step with CUDA events around every engine call (bts_b200.conv trace): the dominant
    kernel's nominal FLOPs over all its launches in the step / the sum of their durations (FLOP-weighted by construction)."""
    conv.set_trace(True)
    try:
        step_fn()
        rep = conv.trace_report()
    finally:
        conv.set_trace(False)
    agg = {}
    for t, n, (kind, desc), fl in rep:
        g = {"fwd": "conv", "dgrad": "conv", "wgrad": "wgrad"}.get(kind)
        if g is None:
            continue
        a = agg.setdefault(g, {"ms": 0.0, "launches": 0, "flops": 0.0, "layers": []})
        a["ms"] += t
        a["launches"] += n
        a["flops"] += fl
        a["layers"].append((t, n, kind, desc, fl))
    peak = pk_tf32["tf32_tflops_sustained"] / 3.0
    out = {}
    for g, a in agg.items():
        ach = a["flops"] / a["ms"] / 1e9 if a["ms"] > 0 else 0.0
        top = sorted(a["layers"], reverse=True)[:6]
        out[g] = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                  "launches_per_step": a["launches"], "ms_per_step": a["ms"],
                  "avg_launch_ms": a["ms"] / max(1, a["launches"]), "algorithmic_flops_per_step": a["flops"],
                  "peak_source": "parity mode 3xTF32: TF32 GEMM peak measured live by this run (sustained, the kernel is timed "
                                 "inside a long step) / 3 products",
                  "top_layers": [{"kind": k, "layer": d, "calls": n, "ms": round(t, 3), "tflops": round(fl / t / 1e9, 1)}
                                 for t, n, k, d, fl in top]}
    return out


OUTPUT_NAMES = ("depth_8x8_scaled", "depth_4x4_scaled", "depth_2x2_scaled", "reduc1x1", "final_depth")
DUMP_CAP = 1 << 21        # elements per dumped array: at most 7 arrays of 8 MiB (float32), under 64 MiB in all


def dump_outputs(path, keep, model, train, torch):
    """--dump-outputs: what the last timed step computed, as <path>/<name>.npy in float32 -- the model's five outputs and,
    for a training step, the loss, the parameters after the optimizer step and their gradients (each flattened in
    model.parameters() order, frozen parameters have no gradient).  An array of more than DUMP_CAP elements is replaced
    by the same fixed sample every run: the elements at the sorted first DUMP_CAP indices of a seed-0 permutation."""
    import numpy as np
    arrays = dict(zip(OUTPUT_NAMES, keep["out"]))
    if train:
        arrays["loss"] = keep["loss"]
        ps = list(model.parameters())
        arrays["params"] = torch.cat([q.detach().reshape(-1) for q in ps])
        arrays["grads"] = torch.cat([q.grad.reshape(-1) for q in ps if q.grad is not None])
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_CAP:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_CAP].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def _run_ours(args):
    import torch
    import torch.distributed as dist
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import bts
    from bts_b200 import _lib, conv, fused
    _lib.lib()                                   # fail loudly if the CUDA library is missing
    selfcheck = None
    if not args.no_selfcheck:
        if rank == 0:
            selfcheck = run_selfcheck()
            flags = [1 if selfcheck[f][0] else 0 for f in SELFCHECK_FEATURES]
        else:
            flags = [1] * len(SELFCHECK_FEATURES)
        if world > 1:
            ft = torch.tensor(flags, device=dev, dtype=torch.int32)
            dist.broadcast(ft, 0)
            flags = [int(v) for v in ft.tolist()]
        lean_ok, onepass_ok, bnb_ok, adam_ok = [bool(v) for v in flags]
        _lib.lib().bts_conv_set_issue_mode(1 if lean_ok else 0)
        fused.BN_ONEPASS = fused.BN_ONEPASS and onepass_ok
        fused.EPI_BNBWD = fused.EPI_BNBWD and bnb_ok      # off by default (measured slower, bts_b200/fused.py); opt-in via env
        if not adam_ok:
            args.optimizer = "torch"
    torch.backends.cudnn.benchmark = True        # bts_main.py:402
    torch.manual_seed(0)
    p = types.SimpleNamespace(encoder=cfg["encoder"], max_depth=cfg["max_depth"], dataset=cfg["dataset"], bts_size=512,
                              pretrained=False)
    model = bts.BtsModel(p)
    train = cfg["train"]
    if train:
        model.train()
        model.decoder.apply(bts.weights_init_xavier)
        freeze_like_set_misc(model)
    else:
        model.eval()
    model.to(dev)
    red = bcast = None
    if world > 1 and train and args.reducer == "ddp":
        # exactly the reference's wrap.  bts_main.py:352 passes find_unused_parameters=True because the ResNet/ResNeXt
        # encoders keep a never-used `fc` (SURVEY Q11); DenseNet-161 has no unused parameter, so the extra autograd
        # traversal is switched off here.
        unused = any(k.startswith("encoder.base_model.fc") for k, _ in model.named_parameters())
        model = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], find_unused_parameters=unused,
                                                          gradient_as_bucket_view=True)
    elif world > 1 and train:
        # B200-native schedule (bts_b200/dist.py): ONE all-reduce of the flat gradient vector after backward and one flat
        # broadcast of rank 0's BatchNorm buffers before forward -- the same two collectives DDP issues (C1, C3 of SURVEY
        # 2.5), un-bucketed: the persistent 1-CTA-per-SM conv kernels leave NCCL no SM to overlap on anyway.
        from bts_b200 import dist as D
        with torch.no_grad():
            ps = list(model.parameters())
            flat = torch.cat([q.detach().reshape(-1) for q in ps])
            dist.broadcast(flat, 0)                                      # C2: initial parameter broadcast
            o = 0
            for q in ps:
                q.copy_(flat[o:o + q.numel()].view_as(q))
                o += q.numel()
            del flat
        red = D.FlatGradReducer(model.parameters())
        bcast = D.FlatBufferBroadcaster(model)
    opt = make_optimizer(model, torch, fused=(args.optimizer == "fused")) if train else None
    crit = bts.silog_loss(0.85)
    B = cfg["B"]
    img, focal, gt = synth_batch(cfg, B, 1 + rank, dev)
    himg, hfocal, hgt = synth_batch(cfg, B, 1 + rank, pin=True)
    total_steps = 10000

    keep = {} if args.dump_outputs else None     # the last step's outputs and loss, for --dump-outputs

    def graph_loss(out, g):
        if keep is not None:
            keep["out"] = out                    # the capture calls this last: these are the graph's static outputs
        return crit(out[4], g, g > cfg["thr"])

    graphed = None
    graph_note = "off"
    if train and args.graph != "off" and args.reducer != "ddp":
        # forward + loss + backward of one step as ONE CUDA graph (bts_b200/graph.py); collective + optimizer stay eager
        try:
            from bts_b200.graph import GraphedTrainStep
            graphed = GraphedTrainStep(model, graph_loss, ((img, focal), (gt,)))
            graph_note = "fwd+loss+bwd captured in one CUDA graph (%d native launches per replay)" % graphed.launches_per_replay
        except Exception as e:
            if args.graph == "on":
                raise
            graphed = None
            graph_note = "capture failed (%s: %s) -> eager launches" % (type(e).__name__, str(e)[:120])
            for q in model.parameters():
                q.grad = None
            torch.cuda.synchronize()

    def step(i, x, f, g):
        if not train:
            with torch.no_grad():
                out = model(x, f)
            if keep is not None:
                keep["out"] = out
            return out[4].sum()
        if bcast is not None:
            bcast.broadcast(0)
        if graphed is not None:
            loss = graphed((x, f), (g,))
        else:
            opt.zero_grad()
            out = model(x, f)
            loss = crit(out[4], g, g > cfg["thr"])
            loss.backward()
            if keep is not None:
                keep["out"] = out
        if keep is not None:
            keep["loss"] = loss
        if red is not None:
            red.reduce(inplace=graphed is not None)
        lr = (1e-4 - 1e-5) * (1 - i / total_steps) ** 0.9 + 1e-5
        for grp in opt.param_groups:
            grp["lr"] = lr
        opt.step()
        return loss

    def timed(fn, K, Wm):
        if world > 1:
            # exercise the collectives of the bracket (barrier, MAX all-reduce) once BEFORE the warm-up steps: their first use
            # sets up NCCL state lazily, and at 8 GPUs the aftermath landed in the first timed step of one rank (+90-120 ms on
            # the max-over-ranks span, absent from rank 0's per-step events and from the second timed() call)
            dist.barrier()
            dist.all_reduce(torch.zeros(1, device=dev), op=dist.ReduceOp.MAX)
            torch.cuda.synchronize()
        for i in range(Wm):
            fn(i)
        # rank 0 forks nvidia-smi BEFORE the barrier: the fork of a process with a CUDA context costs tens of ms, and with
        # N > 1 every other rank would wait for rank 0 in the first all-reduce -- inside ITS timed span (measured: +86 ms on
        # the max-over-ranks span of a 10-step run at 8 GPUs)
        sampler = ClockSampler(local) if rank == 0 else None
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if sampler:
            sampler.mark()
        l0 = _lib.launches
        st = torch.cuda.current_stream()
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        marks[0].record(st)
        for i in range(K):
            fn(Wm + i)
            marks[i + 1].record(st)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([marks[0].elapsed_time(marks[K])], device=dev)
        if world > 1:
            spans = [torch.zeros(1, device=dev) for _ in range(world)]
            dist.all_gather(spans, ms)
            timed.rank_spans_ms = [round(float(t), 2) for t in spans]      # reported: shows rank skew / one-off stalls
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        per = sorted(marks[i].elapsed_time(marks[i + 1]) for i in range(K))
        clocks = sampler.stop() if sampler else None
        return float(ms), _lib.launches - l0, clocks, per

    K, Wm = args.steps, max(args.warmup, 3)
    ms, launches, clocks, per = timed(lambda i: step(i, img, focal, gt), K, Wm)
    rank_spans = getattr(timed, "rank_spans_ms", None)

    def e2e_step(i):
        if graphed is not None:                  # H2D straight into the graph's static input buffers
            return float(step(i, himg, hfocal, hgt).detach())
        x = himg.to(dev, non_blocking=True)
        f = hfocal.to(dev, non_blocking=True)
        g = hgt.to(dev, non_blocking=True)
        return float(step(i, x, f, g).detach())  # D2H read of the loss (bts_main.py:463) / of the result every step

    ms_e, _, _, per_e = timed(e2e_step, K, 1)
    if keep is not None and rank == 0:
        dump_outputs(args.dump_outputs, keep, model, train, torch)
    h2d = himg.numel() * 4 + hfocal.numel() * 8 + hgt.numel() * 4

    pk = peaks()
    res = {
        "metric": cfg["metric"], "value": world * B * K / (ms / 1e3), "unit": "images/s",
        "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "global_batch": world * B, "parallelism": "dp%d" % world,
                   "collective": ("none" if world == 1 or not train else
                                  ("torch DDP (25 MB buckets, overlapped)" if args.reducer == "ddp" else
                                   "one NCCL all-reduce (AVG) of the flat gradient vector per step + one flat buffer broadcast")),
                   "l2": "no explicit flush: per-step working set (saved activations, GBs) >> 126 MB L2",
                   "precision": "3xTF32 split on tcgen05 (fp32-grade, parity mode)",
                   "cuda_graph": graph_note,
                   "optimizer": ("bts_b200.optim.FusedAdamW (one multi-tensor kernel + one re-pack launch)"
                                 if args.optimizer == "fused" else "torch.optim.AdamW") if train else "none"},
        "e2e": {"value": world * B * K / (ms_e / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e / K, "ms_per_step_median": statistics.median(per_e)},
        "repeats": {"ms_per_step_median": statistics.median(per), "ms_per_step_min": per[0], "ms_per_step_max": per[-1],
                    "n": K, "note": "rank-0 per-step CUDA-event durations inside the timed region",
                    "rank_spans_ms": rank_spans},
        "gpu_launches": launches, "clocks": clocks,
    }
    if selfcheck is not None:
        res["selfcheck"] = {f: {"enabled": bool(selfcheck[f][0]), "detail": selfcheck[f][1]} for f in SELFCHECK_FEATURES}
    if rank == 0:
        res["roofline_step"] = {"bound": "tensor", "achieved": res["value"] / world * cfg["gflop"] / 1e3,
                                "unit": "TFLOP/s per GPU (nominal conv FLOPs %.1f GFLOP/img)" % cfg["gflop"]}
        if world == 1 and not args.no_roofline:
            try:
                live = tf32_peak(torch)
            except Exception as e:                 # an evidence leg must never cost the bench line
                live = {"tf32_tflops": pk["bf16_tflops"] / 2.0, "tf32_tflops_sustained": pk["bf16_tflops_sustained"] / 2.0,
                        "how": "FAILED (%s): derived bf16/2 from %s" % (e, pk["source"])}
            res["peaks_live"] = dict(live, hbm_gbs=pk["hbm_gbs"], bf16_tflops=pk["bf16_tflops"],
                                     bf16_tflops_sustained=pk["bf16_tflops_sustained"], hbm_bf16_source=pk["source"])
            roof3 = live["tf32_tflops_sustained"] / 3.0
            res["roofline_step"].update(peak=roof3, frac=res["roofline_step"]["achieved"] / roof3,
                                        peak_note="parity-grade 3xTF32 = TF32 GEMM peak measured live (sustained) / 3")
            if train:
                try:
                    def eager_step():                       # the traced step runs eagerly (CUDA events around every call)
                        for q in model.parameters():
                            q.grad = None
                        o = model(img, focal)
                        crit(o[4], gt, gt > cfg["thr"]).backward()
                    rl = conv_rooflines(torch, conv, eager_step, live)
                    if "conv" in rl:
                        res["roofline"] = dict(rl["conv"], kernel="conv_tc_kernel (tcgen05 implicit GEMM: every conv forward and "
                                                                  "dgrad of the step), all launches of one real training step",
                                               # ncu --set full, profiles/r02_conv_db1_final.ncu-rep: dense 3x3 192->48 @88x176x16
                                               # (the most frequent shape of the kernel), one launch: 191.1 MB read + 33.8 MB
                                               # written vs 238.0 MB algorithmic (input 190.3 + output 47.6 + weights 0.08)
                                               traffic=224.9e6, traffic_unit="bytes, ONE launch of the dense 3x3 192->48 layer (ncu "
                                                                             "capture profiles/r02_conv_db1_final.ncu-rep; algorithmic "
                                                                             "238 MB: no re-reads from DRAM; l1tex 82 %, tensor pipe 33 %)")
                    if "wgrad" in rl:
                        res["roofline_wgrad"] = dict(rl["wgrad"], kernel="wgrad kernels (tcgen05, MN-major operands), all launches "
                                                                         "of one real training step",
                                                     # profiles/r02_wgrad2_db1_final.ncu-rep (dense 3x3 wgrad): 243.0 MB read + 3.8 MB written
                                                     # vs 238.0 MB algorithmic (x 190.3 + dY 47.6); tensor pipe 72.6 %
                                                     traffic=246.8e6, traffic_unit="bytes, ONE launch of the dense 3x3 192->48 wgrad (ncu, "
                                                                                   "profiles/r02_wgrad2_db1_final.ncu-rep; algorithmic 238 MB)")
                except Exception as e:
                    res["roofline"] = {"error": "%s: %s" % (type(e).__name__, e)}
            del model, opt
            torch.cuda.empty_cache()
            if not args.no_lpg:
                res["roofline_lpg"] = lpg_roofline(torch, dev, pk)
            if "roofline" not in res and "roofline_lpg" in res:
                res["roofline"] = res["roofline_lpg"]          # forward-only config: the HBM-bound LPG pair
            if not args.no_gpu_baseline:
                try:
                    res["gpu_baseline"] = gpu_reference_steps(cfg, torch, dev)
                except Exception as e:
                    res["gpu_baseline"] = {"error": "%s: %s" % (type(e).__name__, e)}
            if not args.no_cpu:
                res["cpu_baseline"] = cpu_reference_steps(cfg, 3, 1, budget_s=150.0)
    return res, rank, (dist if world > 1 else None)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config if args.config in CONFIGS else "K16"]
    with StdoutToStderr():
        r = cpu_reference_steps(cfg, args.steps, args.warmup)
    res = {"impl": "reference", "metric": cfg["metric"], "value": r["value"],
           "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": cfg["workload"] + "; CPU sample: " + r["sample"]},
           "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
           "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (launches per point for --config LPG)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="K16", choices=sorted(CONFIGS) + ["LPG"])
    ap.add_argument("--reducer", default="flat", choices=["flat", "ddp"],
                    help="N>1: flat = one all-reduce of the flat gradient vector (bts_b200/dist.py); ddp = torch DDP as bts_main.py")
    ap.add_argument("--optimizer", default="fused", choices=["fused", "torch"],
                    help="fused = bts_b200.optim.FusedAdamW (default), torch = torch.optim.AdamW exactly as bts_main.py")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="capture fwd+loss+bwd of the train step in one CUDA graph (auto: fall back to eager if capture fails)")
    ap.add_argument("--no-selfcheck", action="store_true", help="skip the pre-flight parity check of the round-2 fast paths")
    ap.add_argument("--selfcheck-child", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--no-lpg", action="store_true", help="skip the LPG roofline microbench")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the torch-eager/cuDNN reference leg")
    ap.add_argument("--no-roofline", action="store_true", help="skip every evidence leg (peaks, traced step, LPG, baselines)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config == "LPG"):
        ap.error("--dump-outputs writes the outputs of our model's step: not with --impl reference or --config LPG")
    if args.selfcheck_child is not None:
        selfcheck_child(set(args.selfcheck_child.split(",")))
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
