"""MobileNetV2 encoder (`mobilenetv2_bts`) on one GPU, as one JSON line:

  train   one train step (fwd + silog + bwd + FusedAdamW, fwd+loss+bwd captured by GraphedTrainStep) at 352x704, batch 16,
          KITTI-shaped synthetic inputs -- ours vs the unmodified reference under torch-eager + cuDNN (fp32 and PyTorch's
          TF32 default), both through bench.gpu_reference_steps
  eval    eval-mode forward at 416x544, batch 1
  dw      each depthwise kernel (fwd with the BN+ReLU6 prologue and the statistics epilogue, as the train step runs it;
          dgrad; wgrad) at the 176x352, 88x176 and 44x88 maps of the K16 shape, batch 16: achieved GB/s from algorithmic
          bytes (every tensor read or written once), against a device-to-device copy measured in the same run; L2 is
          overwritten between timed launches
GPU name and power limit are read in the same run.  Usage: python tools/mobilenet_bench.py [--steps 20 --warmup 5]
"""
import argparse
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

TRAIN = dict(encoder="mobilenetv2_bts", H=352, W=704, B=16, dataset="kitti", max_depth=80.0, focal=721.5377, valid=0.2,
             thr=1.0, train=True)
EVAL = dict(encoder="mobilenetv2_bts", H=416, W=544, B=1, dataset="nyu", max_depth=10.0, focal=518.8579, valid=0.95,
            thr=0.1, train=False)
# (input map, channels, stride) of the depthwise layers at 352x704: block 1 / 2 read the 176x352 map, blocks 3 / 4 the
# 88x176 map, blocks 5-7 the 44x88 map
DW_LAYERS = [((176, 352), 32, 1), ((176, 352), 96, 2), ((88, 176), 144, 1), ((88, 176), 144, 2), ((44, 88), 192, 1),
             ((44, 88), 192, 2)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def _model(cfg, torch, dev):
    import bts
    p = types.SimpleNamespace(encoder=cfg["encoder"], max_depth=cfg["max_depth"], dataset=cfg["dataset"], bts_size=512,
                              pretrained=False)
    torch.manual_seed(0)
    m = bts.BtsModel(p)
    m.decoder.apply(bts.weights_init_xavier)
    return m.to(dev)


def _time(torch, fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def ours_train(torch, dev, steps, warmup):
    import bts
    from bts_b200.graph import GraphedTrainStep
    m = _model(TRAIN, torch, dev).train()
    opt = bench.make_optimizer(m, torch, fused=True)
    img, focal, gt = bench.synth_batch(TRAIN, TRAIN["B"], 1, dev)
    crit = bts.silog_loss(0.85)
    graphed = GraphedTrainStep(m, lambda out, g: crit(out[4], g, g > TRAIN["thr"]), ((img, focal), (gt,)))

    def step():
        graphed((img, focal), (gt,))
        opt.step()

    ms = _time(torch, step, steps, warmup)
    del m, opt, graphed
    torch.cuda.empty_cache()
    return {"value": TRAIN["B"] / (ms / 1e3), "unit": "images/s", "ms_per_step": ms}


def ours_eval(torch, dev, steps, warmup):
    m = _model(EVAL, torch, dev).eval()
    img, focal, _ = bench.synth_batch(EVAL, 1, 1, dev)

    def fwd():
        with torch.no_grad():
            m(img, focal)

    ms = _time(torch, fwd, steps, warmup)
    del m
    torch.cuda.empty_cache()
    return {"value": 1.0 / (ms / 1e3), "unit": "images/s", "ms_per_forward": ms}


def _kernel_ms(torch, fn, flush, reps):
    """median of `reps` launches, each timed alone after L2 has been overwritten"""
    ts = []
    for i in range(reps + 2):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if i >= 2:
            ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def dw_kernels(torch, dev, reps):
    from bts_b200 import glue
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)           # 256 MB > the 126 MB L2
    src = torch.empty(1 << 28, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    copy_gbs = 2 * src.numel() / (_kernel_ms(torch, lambda: dst.copy_(src), flush, reps) * 1e6)
    out = {"copy_gbs": copy_gbs, "copy_what": "torch copy_ of 256 MB device to device, read + write bytes over time",
           "layers": []}
    del src, dst
    B = 16
    g = torch.Generator(device=dev).manual_seed(0)
    for (H, W), C, s in DW_LAYERS:
        Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
        x = torch.randn(B, C, H, W, device=dev, generator=g).contiguous(memory_format=torch.channels_last)
        gy = torch.randn(B, C, Ho, Wo, device=dev, generator=g).contiguous(memory_format=torch.channels_last)
        w = torch.randn(C, 1, 3, 3, device=dev, generator=g)
        st = torch.stack([torch.ones(C, device=dev), torch.zeros(C, device=dev), torch.zeros(C, device=dev),
                          torch.ones(C, device=dev)])
        big, small = B * H * W * C * 4, B * Ho * Wo * C * 4
        row = {"map": "%dx%d" % (H, W), "C": C, "stride": s}
        for kind, fn, nbytes in (("fwd", lambda: glue.dw_fwd(x, w, s, pre=st, stats=True), big + small),
                                 ("dgrad", lambda: glue.dw_dgrad(gy, w, s, H, W), small + big),
                                 ("wgrad", lambda: glue.dw_wgrad(x, gy, w, s, pre=st), big + small)):
            ms = _kernel_ms(torch, fn, flush, reps)
            row[kind] = {"us": ms * 1e3, "gbs": nbytes / (ms * 1e6), "of_copy": nbytes / (ms * 1e6) / copy_gbs}
        out["layers"].append(row)
        del x, gy
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20, help="timed launches per depthwise kernel")
    ap.add_argument("--no-reference", action="store_true", help="skip the torch-eager + cuDNN reference leg")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mobilenet_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "workload": "mobilenetv2_bts, random-init weights, synthetic inputs (bench.synth_batch)"}
    res["dw"] = dw_kernels(torch, dev, args.reps)
    res["train_352x704_b16"] = {"ours": ours_train(torch, dev, args.steps, args.warmup)}
    if not args.no_reference:
        res["train_352x704_b16"]["reference"] = bench.gpu_reference_steps(TRAIN, torch, dev,
                                                                         args.steps, args.warmup)
    res["eval_416x544_b1"] = {"ours": ours_eval(torch, dev, args.steps * 5, args.warmup)}
    if not args.no_reference:
        res["eval_416x544_b1"]["reference"] = bench.gpu_reference_steps(EVAL, torch, dev, args.steps * 5, args.warmup)
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
