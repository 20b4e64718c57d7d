"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the UNMODIFIED reference (its pytorch/ directory,
found by oracle/ref_shim.py: $BTS_REFERENCE_DIR or the copy `make -C oracle` leaves in oracle/_ref/) on seeded inputs,
on the CPU, fp32.

    python oracle/make_golden.py [core] [models] [lpg_shapes] [io]      # no argument: every group
The committed fixtures are what pins oracle/bts_oracle.py and the CUDA path to the reference; the tests read only them.
"""
import ast
import os
import random
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from ref_shim import load_reference  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")


def head_planes(B, h, w, max_depth, gen):
    """Plane coefficients through the real head parametrisation (BASELINE.md LPG-u inputs)."""
    z = torch.randn(B, 3, h, w, generator=gen)
    th = torch.sigmoid(z[:, 0]) * np.pi / 3
    ph = torch.sigmoid(z[:, 1]) * np.pi * 2
    d = torch.sigmoid(z[:, 2]) * max_depth
    return torch.stack([torch.sin(th) * torch.cos(ph), torch.sin(th) * torch.sin(ph), torch.cos(th), d], 1).contiguous()


def core_fixtures(R):
    # ---- LPG: forward + autograd gradient, r = 2, 4, 8 (pytorch/bts.py:124-146)
    for r in (2, 4, 8):
        gen = torch.Generator().manual_seed(100 + r)
        plane = head_planes(2, 5, 6, 10.0, gen).requires_grad_(True)
        mod = R.local_planar_guidance(r)
        depth = mod(plane, torch.tensor([518.8579, 518.8579]))
        dy = torch.randn(depth.shape, generator=gen)
        depth.backward(dy)
        np.savez_compressed(os.path.join(OUT, "lpg_r%d.npz" % r), plane=plane.detach().numpy(),
                            depth=depth.detach().numpy(), dy=dy.numpy(), dplane=plane.grad.numpy())

    # ---- reduction_1x1 (non-final and final) (pytorch/bts.py:83-122)
    gen = torch.Generator().manual_seed(7)
    torch.manual_seed(7)
    for final in (False, True):
        mod = R.reduction_1x1(32, 16, 10.0, is_final=final)
        x = torch.randn(2, 32, 6, 7, generator=gen)
        y = mod(x)
        d = {"x": x.numpy(), "y": y.detach().numpy()}
        d.update({"sd." + k: v.numpy() for k, v in mod.state_dict().items()})
        np.savez_compressed(os.path.join(OUT, "reduc_%s.npz" % ("final" if final else "plane")), **d)

    # ---- silog_loss forward + autograd gradient (pytorch/bts.py:41-48)
    gen = torch.Generator().manual_seed(11)
    est = (torch.rand(2, 1, 16, 24, generator=gen) * 79 + 1).requires_grad_(True)
    gt = torch.rand(2, 1, 16, 24, generator=gen) * 80
    gt = torch.where(torch.rand(2, 1, 16, 24, generator=gen) < 0.3, gt, torch.zeros_like(gt))
    mask = gt > 1.0
    loss = R.silog_loss(0.85).forward(est, gt, mask)
    loss.backward()
    np.savez_compressed(os.path.join(OUT, "silog.npz"), est=est.detach().numpy(), gt=gt.numpy(),
                        mask=mask.numpy(), loss=loss.detach().numpy(), dest=est.grad.numpy())

    # ---- whole decoder `bts` (pytorch/bts.py:148-266), small widths, eval and train mode
    feat = [8, 8, 16, 24, 40]
    for dataset, max_depth in (("kitti", 80.0), ("nyu", 10.0)):
        torch.manual_seed(3)
        params = types.SimpleNamespace(max_depth=max_depth, dataset=dataset)
        dec = R.bts(params, feat, num_features=128)
        dec.apply(R.weights_init_xavier)
        gen = torch.Generator().manual_seed(5)
        with torch.no_grad():      # non-trivial BN affine / running stats
            for m in dec.modules():
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.weight.copy_(torch.rand(m.weight.shape, generator=gen) + 0.5)
                    m.bias.copy_(torch.randn(m.bias.shape, generator=gen) * 0.1)
                    m.running_mean.copy_(torch.randn(m.bias.shape, generator=gen) * 0.1)
                    m.running_var.copy_(torch.rand(m.bias.shape, generator=gen) + 0.5)
        H = W = 64
        B = 2
        feats = [torch.randn(B, feat[i], H >> (i + 1), W >> (i + 1), generator=gen) for i in range(5)]
        focal = torch.tensor([721.5377, 707.0912])
        d = {"focal": focal.numpy(), "feat_channels": np.array(feat), "num_features": np.array(128),
             "max_depth": np.array(max_depth)}
        d.update({"feat%d" % i: f.numpy() for i, f in enumerate(feats)})
        d.update({"sd." + k: v.clone().numpy() for k, v in dec.state_dict().items()})
        dec.eval()
        with torch.no_grad():
            outs = dec(feats, focal)
        d.update({"eval_out%d" % i: o.numpy() for i, o in enumerate(outs)})
        dec.train()
        with torch.no_grad():
            outs = dec(feats, focal)
        d.update({"train_out%d" % i: o.numpy() for i, o in enumerate(outs)})
        d.update({"sd_after." + k: v.numpy() for k, v in dec.state_dict().items() if "running" in k})
        np.savez_compressed(os.path.join(OUT, "decoder_%s.npz" % dataset), **d)


MODEL_ENCODERS = ("densenet121_bts", "resnext50_bts", "mobilenetv2_bts")
MODEL_SAMPLE = 512        # output elements stored per output tensor (plus exact float64 sums of the whole tensor)


def seeded_state_dict(model, seed=0):
    """Weights for a whole-model comparison that depend only on the state_dict keys and shapes, not on how a model
    initialises itself: filled in sorted key order from one seeded generator.  Conv / linear weights are normal with
    Glorot's variance 2 / (fan_in + fan_out): with it every output of all three encoder families stays well inside the
    sigmoid's range in eval and train mode, where the fp32 differences of another thread count or CPU stay ~100x below
    the test's bar (saturated outputs amplify them).  BatchNorm scales and running variances are U(0.75, 1.25); shifts,
    biases and running means N(0, 0.05^2)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, v in sorted(model.state_dict().items()):
        if not v.is_floating_point():
            sd[k] = v.clone()
        elif k.endswith("running_mean") or (v.dim() == 1 and k.endswith("bias")):
            sd[k] = torch.randn(v.shape, generator=g) * 0.05
        elif k.endswith("running_var") or v.dim() == 1:
            sd[k] = torch.rand(v.shape, generator=g) * 0.5 + 0.75
        else:
            sd[k] = torch.randn(v.shape, generator=g) * (2.0 / (v[0].numel() + v.shape[0] * v[0, 0].numel())) ** 0.5
    return sd


def model_inputs():
    """(mode, x, focal) of the whole-model comparison: eval on one image, then train (batch statistics) on two."""
    x = torch.randn(1, 3, 64, 96, generator=torch.Generator().manual_seed(1))
    return [("eval", x, torch.tensor([518.8579])),
            ("train", torch.cat([x, x.flip(3)], 0), torch.tensor([518.8579, 518.8579]))]


def model_fixtures(R):
    """Whole BtsModel (DenseNet / ResNeXt / MobileNetV2 encoders, pytorch/bts.py:273-331) under seeded_state_dict:
    a fixed seeded sample of every output plus its float64 sum and absolute sum, and the state_dict keys and shapes."""
    for enc in MODEL_ENCODERS:
        p = types.SimpleNamespace(encoder=enc, max_depth=10.0, dataset="nyu", bts_size=512)
        torch.manual_seed(0)
        ref = R.BtsModel(p)
        ref.load_state_dict(seeded_state_dict(ref), strict=True)
        d = {"keys": np.array(sorted("%s:%s" % (k, "x".join(map(str, v.shape))) for k, v in ref.state_dict().items()))}
        for mode, x, focal in model_inputs():
            getattr(ref, mode)()
            with torch.no_grad():
                outs = ref(x, focal)
            n = outs[0].numel()
            idx = torch.randperm(n, generator=torch.Generator().manual_seed(2))[:MODEL_SAMPLE].sort().values
            d[mode + "_idx"] = idx.numpy().astype(np.int32)
            for i, o in enumerate(outs):
                assert o.numel() == n
                v = o.reshape(-1).double()
                d["%s_out%d" % (mode, i)] = o.reshape(-1)[idx].numpy()
                d["%s_out%d_sum" % (mode, i)] = np.float64(v.sum())
                d["%s_out%d_abssum" % (mode, i)] = np.float64(v.abs().sum())
        np.savez_compressed(os.path.join(OUT, "model_%s.npz" % enc), **d)


LPG_SHAPE_CASES = 12


def lpg_shape_fixtures(R):
    """The reference LPG module on randomly drawn shapes (B 1-3, h 1-6, w 1-7, r 2/4/8) and plane seeds."""
    rng = np.random.RandomState(12)
    cases = np.stack([rng.randint(1, 4, LPG_SHAPE_CASES), rng.randint(1, 7, LPG_SHAPE_CASES),
                      rng.randint(1, 8, LPG_SHAPE_CASES), rng.choice([2, 4, 8], LPG_SHAPE_CASES),
                      rng.randint(0, 10 ** 6, LPG_SHAPE_CASES)], 1)
    d = {"cases": cases}
    for j, (B, h, w, r, seed) in enumerate(cases.tolist()):
        plane = head_planes(B, h, w, 10.0, torch.Generator().manual_seed(seed))
        depth = R.local_planar_guidance(r)(plane, torch.full((B,), 518.8579))
        d["depth%d" % j] = depth.reshape(B, h * r, w * r).numpy()
    np.savez_compressed(os.path.join(OUT, "lpg_shapes.npz"), **d)


IO_SEEDS = 6


def io_fixtures(R):
    """compute_errors (pytorch/bts_main.py:144-165, extracted by ast because the script parses argv at import) and the
    training-loader transform DataLoadPreprocess.random_crop / train_preprocess / ToTensor (pytorch/bts_dataloader.py)
    with the random module and numpy seeded per draw."""
    from ref_shim import REFERENCE_DIR
    src = open(os.path.join(REFERENCE_DIR, "bts_main.py")).read()
    fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "compute_errors"][0]
    ns = {"np": np}
    exec(compile(ast.Module([fn], []), "bts_main.compute_errors", "exec"), ns)
    rng = np.random.RandomState(0)
    gt = rng.uniform(0.5, 70, 5000).astype(np.float32)
    pred = (gt * rng.uniform(0.6, 1.6, 5000)).astype(np.float32)
    d = {"compute_errors": np.array(ns["compute_errors"](gt, pred), dtype=np.float64)}

    sys.path.insert(0, REFERENCE_DIR)
    import bts_dataloader as D
    H, W = 32, 32
    for dataset, div in (("nyu", 1000.0), ("kitti", 256.0)):
        ds = D.DataLoadPreprocess.__new__(D.DataLoadPreprocess)
        ds.args = types.SimpleNamespace(dataset=dataset)
        rng = np.random.RandomState(1)
        img_u8 = rng.randint(0, 256, (40, 56, 3)).astype(np.uint8)
        dep_u16 = rng.randint(0, 60000, (40, 56)).astype(np.uint16)
        images, depths = [], []
        for seed in range(IO_SEEDS):
            random.seed(seed)
            np.random.seed(seed)
            image = np.asarray(img_u8, dtype=np.float32) / 255.0
            depth = np.expand_dims(np.asarray(dep_u16, dtype=np.float32), 2) / div
            ci, cd = ds.random_crop(image, depth, H, W)
            ri, rd = ds.train_preprocess(ci, cd)
            sample = D.ToTensor("train")({"image": ri, "depth": rd, "focal": 1.0})
            images.append(sample["image"].numpy())
            depths.append(sample["depth"].numpy())
        d[dataset + "_image"] = np.stack(images)
        d[dataset + "_depth"] = np.stack(depths)
    np.savez_compressed(os.path.join(OUT, "io_reference.npz"), **d)


FIXTURES = {"core": core_fixtures, "models": model_fixtures, "lpg_shapes": lpg_shape_fixtures, "io": io_fixtures}


def main(names):
    os.makedirs(OUT, exist_ok=True)
    R = load_reference()
    torch.set_num_threads(4)
    for name in names or FIXTURES:
        FIXTURES[name](R)
    print("golden fixtures written to", os.path.abspath(OUT))
    for f in sorted(os.listdir(OUT)):
        print("  %-24s %8d bytes" % (f, os.path.getsize(os.path.join(OUT, f))))


if __name__ == "__main__":
    main(sys.argv[1:])
