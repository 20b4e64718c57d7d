"""Property tests of the oracle (CPU, hypothesis): size-independent invariants of the LPG / silog arithmetic, and
agreement with the unmodified reference module on randomly drawn shapes, stored in tests/golden/lpg_shapes.npz (the
reference ships no tests of its own -- SURVEY 4 -- so shapes beyond the other golden vectors are pinned this way)."""
import numpy as np
import torch
from hypothesis import given, settings, strategies as st

import bts_oracle as O
from conftest import head_planes

shapes = st.tuples(st.integers(1, 3), st.integers(1, 6), st.integers(1, 7), st.sampled_from([2, 4, 8]),
                   st.integers(0, 10 ** 6))


@settings(max_examples=25, deadline=None)
@given(shapes)
def test_lpg_is_homogeneous_in_the_plane_distance(s):
    B, h, w, r, seed = s
    plane = head_planes(B, h, w, 10.0, seed=seed)
    d1 = O.lpg_forward(plane, r)
    scaled = plane.clone()
    scaled[:, 3] *= 4.0                                   # power of two: exact in fp32
    assert torch.equal(O.lpg_forward(scaled, r), d1 * 4.0)


@settings(max_examples=15, deadline=None)
@given(shapes)
def test_lpg_of_a_fronto_parallel_plane_is_its_distance(s):
    B, h, w, r, seed = s
    g = torch.Generator().manual_seed(seed)
    dist = torch.rand(B, h, w, generator=g) * 10 + 0.1
    plane = torch.stack([torch.zeros_like(dist), torch.zeros_like(dist), torch.ones_like(dist), dist], 1)
    d = O.lpg_forward(plane, r)
    assert torch.equal(d, dist.repeat_interleave(r, 1).repeat_interleave(r, 2))


@settings(max_examples=15, deadline=None)
@given(shapes)
def test_lpg_backward_is_the_adjoint_of_the_linearised_forward(s):
    B, h, w, r, seed = s
    plane = head_planes(B, h, w, 10.0, seed=seed).double().requires_grad_(True)
    g = torch.Generator().manual_seed(seed + 1)
    dy = torch.randn(B, h * r, w * r, generator=g, dtype=torch.float64)
    (auto,) = torch.autograd.grad(O.lpg_forward(plane, r), plane, dy)
    ours = O.lpg_backward(dy.float(), plane.detach().float(), r).double()
    scale = auto.abs().max().clamp_min(1e-12)
    assert ((ours - auto).abs().max() / scale) < 1e-4


@settings(max_examples=20, deadline=None)
@given(st.integers(0, 10 ** 6), st.floats(0.25, 8.0))
def test_silog_is_invariant_to_a_common_scale(seed, a):
    g = torch.Generator().manual_seed(seed)
    est = torch.rand(2, 1, 9, 11, generator=g) * 20 + 0.5
    gt = torch.rand(2, 1, 9, 11, generator=g) * 20 + 0.5
    mask = torch.rand(2, 1, 9, 11, generator=g) > 0.3
    l1, l2 = O.silog(est, gt, mask, 0.85), O.silog(est * a, gt * a, mask, 0.85)
    assert abs(float(l1) - float(l2)) <= 1e-4 * max(1.0, abs(float(l1)))


def test_lpg_matches_the_live_reference_module_on_random_shapes(golden):
    g = golden("lpg_shapes")
    assert len(g["cases"]) == 12
    for j, (B, h, w, r, seed) in enumerate(g["cases"].tolist()):
        plane = head_planes(B, h, w, 10.0, seed=seed)
        assert np.array_equal(O.lpg_forward(plane, r).numpy(), g["depth%d" % j]), (B, h, w, r, seed)
