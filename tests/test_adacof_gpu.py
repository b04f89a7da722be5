"""GPU parity tests for the AdaCoF warp: libfvfi.so (through the C-ABI / FunctionAdaCoF) against
the CPU oracle and the committed outputs of the reference's own CUDA kernels (tests/golden/)."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import adacof as oa

pytestmark = pytest.mark.gpu

TOL_FWD = 2e-6      # [0,1] frames, softmax weights (north star: 1e-4)
TOL_BWD = 3e-5      # |gout| ~ N(0,1), 3 channels summed


def _dev(*arrs):
    return [torch.from_numpy(a).cuda() for a in arrs]


SHAPES = [(2, 3, 40, 56, 5, 1), (1, 3, 33, 47, 5, 2), (1, 3, 24, 40, 3, 1), (2, 3, 96, 160, 5, 1),
          (1, 3, 70, 130, 7, 2)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("algo", [1, 2, 0])
def test_forward_backward_vs_oracle(shape, algo):
    from fvfi import adacof
    B, C, H, W, F, d = shape
    if algo == 2 and (F - 1) * d > 8:
        pytest.skip("tiled path covers (F-1)*dilation <= 8")
    inp, w, oi, oj, g = oa.synth(B, C, H, W, F, d, seed=11)
    t_inp, t_w, t_oi, t_oj, t_g = _dev(inp, w, oi, oj, g)
    out = adacof.adacof_forward(t_inp, t_w, t_oi, t_oj, d, algo_=algo)
    ref = oa.forward(inp, w, oi, oj, d, threads=4)
    assert np.abs(out.cpu().numpy() - ref).max() <= TOL_FWD
    gin, gw, gi, gj = adacof.adacof_backward(t_g, t_inp, t_w, t_oi, t_oj, d, "zeros", algo_=algo)
    rgw, rgi, rgj = oa.backward(g, inp, w, oi, oj, d, threads=4)
    assert float(gin.abs().max()) == 0.0  # reference semantics (adacof.py:382,445)
    assert np.abs(gw.cpu().numpy() - rgw).max() <= TOL_BWD
    assert np.abs(gi.cpu().numpy() - rgi).max() <= TOL_BWD
    assert np.abs(gj.cpu().numpy() - rgj).max() <= TOL_BWD


@pytest.mark.parametrize("shape", [(2, 3, 40, 56, 5, 1), (2, 3, 96, 160, 5, 1), (3, 3, 37, 52, 5, 1), (1, 3, 9, 36, 5, 1)])
def test_forward_algorithms_agree(shape):
    """The TMA-streamed forward and backward (algo 3; what `auto` picks for F = 5, dilation 1, W % 4 == 0) equals the tiled kernel
    (algo 2) BIT FOR BIT -- same tap order and contractions -- and both match the oracle, including ragged tile edges
    and offsets far outside the staged halo (clamp-to-edge fallback)."""
    from fvfi import adacof
    B, C, H, W, F, d = shape
    inp, w, oi, oj, _ = oa.synth(B, C, H, W, F, d, seed=17)
    oi = (oi * 2.5).astype(np.float32)          # pushes many taps beyond the +-8 halo
    t = _dev(inp, w, oi, oj)
    o3 = adacof.adacof_forward(*t, d, algo_=3)
    o2 = adacof.adacof_forward(*t, d, algo_=2)
    o0 = adacof.adacof_forward(*t, d, algo_=0)
    assert torch.equal(o3, o2) and torch.equal(o0, o3)
    assert np.abs(o3.cpu().numpy() - oa.forward(inp, w, oi, oj, d, threads=4)).max() <= TOL_FWD
    g = torch.randn(o3.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    b3 = adacof.adacof_backward(g, *t, d, "none", algo_=3)
    b2 = adacof.adacof_backward(g, *t, d, "none", algo_=2)
    for x3, x2 in zip(b3[1:], b2[1:]):
        assert torch.equal(x3, x2)
    rg = oa.backward(g.cpu().numpy(), inp, w, oi, oj, d, threads=4)
    for x3, r in zip(b3[1:], rg):
        assert np.abs(x3.cpu().numpy() - r).max() <= TOL_BWD
    with pytest.raises(Exception):
        adacof.adacof_forward(*_dev(*oa.synth(1, 3, 24, 40, 3, 1, seed=1)[:4]), 1, algo_=3)   # F = 3: not applicable


def test_golden_vectors(golden_dir):
    from fvfi import adacof
    files = sorted(glob.glob(os.path.join(golden_dir, "adacof_ref_*.npz")))
    assert files
    for f in files:
        z = np.load(f)
        B, C, H, W, F, d, seed = [int(v) for v in z["shape"]]
        inp, w, oi, oj, g = oa.synth(B, C, H, W, F, d, seed)
        t_inp, t_w, t_oi, t_oj, t_g = _dev(inp, w, oi, oj, g)
        out = adacof.adacof_forward(t_inp, t_w, t_oi, t_oj, d)
        assert np.abs(out.cpu().numpy() - z["out"]).max() <= TOL_FWD
        _, gw, gi, gj = adacof.adacof_backward(t_g, t_inp, t_w, t_oi, t_oj, d, "none")
        assert np.abs(gw.cpu().numpy() - z["gw"]).max() <= TOL_BWD
        assert np.abs(gi.cpu().numpy() - z["gi"]).max() <= TOL_BWD
        assert np.abs(gj.cpu().numpy() - z["gj"]).max() <= TOL_BWD


@pytest.mark.parametrize("shape", [(2, 3, 40, 56, 5, 1), (1, 3, 33, 47, 5, 2), (1, 3, 24, 40, 3, 1)])
def test_vs_reference_cuda_kernels(golden_dir, shape):
    """Every forward / backward algorithm against the outputs of the reference's own CUDA kernels on a B200
    (tests/golden/adacof_ref_*.npz, made by make_adacof_golden.py; inputs regenerated from the stored seed)."""
    from fvfi import adacof
    B, C, H, W, F, d = shape
    files = glob.glob(os.path.join(golden_dir, "adacof_ref_B%d_C%d_H%d_W%d_F%d_D%d_s*.npz" % shape))
    assert len(files) == 1, files
    z = np.load(files[0])
    seed = int(z["shape"][-1])
    inp, w, oi, oj, g = oa.synth(B, C, H, W, F, d, seed)
    t_inp, t_w, t_oi, t_oj, t_g = _dev(inp, w, oi, oj, g)
    ref_out, rgw, rgi, rgj = _dev(z["out"], z["gw"], z["gi"], z["gj"])
    algos = (1, 2, 3, 0) if (F == 5 and d == 1 and W % 4 == 0) else (1, 2, 0)   # 3 = the TMA-streamed kernel the pipeline runs
    for algo in algos:
        out = adacof.adacof_forward(t_inp, t_w, t_oi, t_oj, d, algo_=algo)
        assert float((out - ref_out).abs().max()) <= TOL_FWD
        _, gw, gi, gj = adacof.adacof_backward(t_g, t_inp, t_w, t_oi, t_oj, d, "none", algo_=algo)
        assert float((gw - rgw).abs().max()) <= TOL_BWD
        assert float((gi - rgi).abs().max()) <= TOL_BWD
        assert float((gj - rgj).abs().max()) <= TOL_BWD


def test_edge_cases():
    from fvfi import adacof
    # single pixel, F=1 (no neighbourhood), huge offsets (every tap clamps), ragged sizes
    for (B, C, H, W, F, d) in [(1, 3, 1, 1, 1, 1), (1, 3, 5, 3, 1, 1), (3, 3, 17, 65, 5, 1), (1, 3, 16, 64, 5, 1)]:
        inp, w, oi, oj, g = oa.synth(B, C, H, W, F, d, seed=4)
        oi = (oi * 40).astype(np.float32)
        oj = (oj * -40).astype(np.float32)
        t = _dev(inp, w, oi, oj)
        for algo in (1, 0):
            out = adacof.adacof_forward(*t, d, algo_=algo)
            assert np.abs(out.cpu().numpy() - oa.forward(inp, w, oi, oj, d)).max() <= TOL_FWD
    # channel counts other than 3 (forward only; the reference backward hard-codes 3)
    inp, w, oi, oj, _ = oa.synth(2, 5, 12, 20, 3, 1, seed=8)
    out = adacof.adacof_forward(*_dev(inp, w, oi, oj), 1)
    assert np.abs(out.cpu().numpy() - oa.forward(inp, w, oi, oj, 1)).max() <= TOL_FWD


def test_preconditions_and_errors():
    from fvfi import adacof, FvfiError
    inp, w, oi, oj, g = oa.synth(1, 3, 8, 8, 3, 1, seed=0)
    t_inp, t_w, t_oi, t_oj = _dev(inp, w, oi, oj)
    with pytest.raises(AssertionError):  # shape relation, adacof.py:326-327
        adacof.FunctionAdaCoF.apply(t_inp[:, :, :-1].contiguous(), t_w, t_oi, t_oj, 1)
    with pytest.raises(AssertionError):  # contiguity, adacof.py:329-332
        nc = torch.empty((1, 9, 8, 16), device="cuda")[..., ::2]
        assert nc.shape == t_w.shape and not nc.is_contiguous()
        adacof.FunctionAdaCoF.apply(t_inp, nc, t_oi, t_oj, 1)
    with pytest.raises(NotImplementedError):  # CPU tensors, adacof.py:356-357
        adacof.FunctionAdaCoF.apply(*[torch.from_numpy(x) for x in (inp, w, oi, oj)], 1)
    inp2, w2, oi2, oj2, g2 = oa.synth(1, 2, 8, 8, 3, 1, seed=0)
    with pytest.raises(FvfiError):  # backward needs C == 3
        adacof.adacof_backward(*_dev(g2, inp2, w2, oi2, oj2), 1)


def test_autograd_function_and_true_grad_input():
    from fvfi import adacof
    B, C, H, W, F, d = 1, 3, 20, 36, 5, 1
    inp, w, oi, oj, g = oa.synth(B, C, H, W, F, d, seed=9)
    ts = [t.requires_grad_(True) for t in _dev(inp, w, oi, oj)]
    out = adacof.FunctionAdaCoF.apply(*ts, d)
    out.backward(torch.from_numpy(g).cuda())
    rgw, rgi, rgj = oa.backward(g, inp, w, oi, oj, d)
    assert float(ts[0].grad.abs().max()) == 0.0
    assert np.abs(ts[1].grad.cpu().numpy() - rgw).max() <= TOL_BWD
    assert np.abs(ts[2].grad.cpu().numpy() - rgi).max() <= TOL_BWD
    assert np.abs(ts[3].grad.cpu().numpy() - rgj).max() <= TOL_BWD
    # extension: true gradInput
    t_g, t_inp, t_w, t_oi, t_oj = _dev(g, inp, w, oi, oj)
    gin, _, _, _ = adacof.adacof_backward(t_g, t_inp, t_w, t_oi, t_oj, d, "true")
    ref = oa.grad_input(g, inp.shape, w, oi, oj, d)
    assert np.abs(gin.cpu().numpy() - ref).max() <= 2e-4  # atomics: order-dependent fp32 sums


# (.., 7, 2): the tile form's region needs the > 48 KB shared-memory opt-in; (.., 11, 4): it does not fit at all -> warp-aggregated kernel
@pytest.mark.parametrize("shape", [(2, 3, 40, 56, 5, 1), (1, 3, 33, 47, 5, 2), (1, 3, 24, 40, 3, 1), (1, 3, 17, 70, 5, 1),
                                   (1, 3, 24, 40, 7, 2), (1, 3, 12, 20, 11, 4)])
@pytest.mark.parametrize("offsets", ["iid", "zero", "smooth", "clamped"])
@pytest.mark.parametrize("scatter", ["tile", "warp"])
def test_true_grad_input_warp_aggregated_scatter(shape, offsets, scatter, monkeypatch):
    """gin_mode "true" (extension beyond the reference, which returns zeros), both forms of the scatter: "tile" (default,
    adacof_grad_input_tile: a CTA accumulates its 64 x 16 pixels' contributions in a shared-memory image of the reachable frame
    region and flushes each non-zero sample with one global reduction; offsets beyond the halo go straight to global memory -- the
    "clamped" case) and "warp" (adacof_grad_input_scatter: __match_any_sync groups lanes by target address, one reduction per
    distinct address; FVFI_GIN_SCATTER=warp) equal the serial adjoint of the oracle -- for scattered addresses, identical addresses in
    every lane (zero offsets / clamped far-out offsets: whole warps collapse onto border samples) and smooth fields; ragged widths leave
    inactive lanes in the last warp.  The other three gradients come from the same fast path as mode "none"."""
    from fvfi import adacof
    monkeypatch.setenv("FVFI_GIN_SCATTER", scatter)
    B, C, H, W, F, d = shape
    inp, w, oi, oj, g = oa.synth(B, C, H, W, F, d, seed=23)
    if offsets == "zero":
        oi, oj = np.zeros_like(oi), np.zeros_like(oj)
    elif offsets == "smooth":
        yy, xx = np.meshgrid(np.arange(H, dtype=np.float32), np.arange(W, dtype=np.float32), indexing="ij")
        oi = np.broadcast_to(1.7 * np.sin(yy / 9.0) - 0.4 + 0.002 * xx, oi.shape).astype(np.float32).copy()
        oj = np.broadcast_to(-2.3 * np.cos(xx / 11.0) + 0.3, oj.shape).astype(np.float32).copy()
    elif offsets == "clamped":
        oi, oj = (oi * 60).astype(np.float32), (oj * -60).astype(np.float32)
    t_g, t_inp, t_w, t_oi, t_oj = _dev(g, inp, w, oi, oj)
    gin, gw, gi, gj = adacof.adacof_backward(t_g, t_inp, t_w, t_oi, t_oj, d, "true")
    ref = oa.grad_input(g, inp.shape, w, oi, oj, d)
    scale = max(1.0, float(np.abs(ref).max()))
    assert np.abs(gin.cpu().numpy() - ref).max() <= 2e-5 * scale      # fp32 sums in a different (atomic) order
    _, gw0, gi0, gj0 = adacof.adacof_backward(t_g, t_inp, t_w, t_oi, t_oj, d, "none")
    assert torch.equal(gw, gw0) and torch.equal(gi, gi0) and torch.equal(gj, gj0)
    # adjoint identity <gout, forward(x)> == <gradInput, x> (the forward is linear in the frame)
    x = torch.randn(t_inp.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    lhs = float((t_g.double() * adacof.adacof_forward(x, t_w, t_oi, t_oj, d).double()).sum())
    rhs = float((gin.double() * x.double()).sum())
    assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs))


def test_fused_warp_blend_and_tail():
    from fvfi import adacof
    B, H, W, F, d = 2, 48, 80, 5, 1
    i1, w1, a1, b1, _ = oa.synth(B, 3, H, W, F, d, seed=31)
    i2, w2, a2, b2, _ = oa.synth(B, 3, H, W, F, d, seed=32)
    occ = np.random.default_rng(3).random((B, 1, H, W), dtype=np.float32)
    t1 = oa.forward(i1, w1, a1, b1, d)
    t2 = oa.forward(i2, w2, a2, b2, d)
    frame, mask = oa.adacofnet_tail(t1, t2, occ, w1, a1, b1, w2, a2, b2)
    dv = _dev(i1, i2, w1, a1, b1, w2, a2, b2, occ)
    g1, g2, gframe, gmask = adacof.adacofnet_warp_blend(*dv, d)
    assert np.abs(g1.cpu().numpy() - t1).max() <= TOL_FWD
    assert np.abs(g2.cpu().numpy() - t2).max() <= TOL_FWD
    assert np.abs(gframe.cpu().numpy() - frame).max() <= TOL_FWD
    assert np.abs(gmask.cpu().numpy() - mask).max() <= 2e-5
    f2, m2 = adacof.adacofnet_tail(g1, g2, dv[8], *dv[2:8])
    assert np.abs(f2.cpu().numpy() - frame).max() <= TOL_FWD
    assert np.abs(m2.cpu().numpy() - mask).max() <= 2e-5


def test_full_size_properties():
    """BASELINE configs[1] size (B=8 x 1088x1920, F=5): size-independent properties.
    (a) zero offsets + one-hot centre weight reproduces the unpadded frame exactly;
    (b) forward is linear in the frame; (c) a random row slab equals the oracle."""
    from fvfi import adacof
    B, C, H, W, F, d = 8, 3, 1088, 1920, 5, 1
    gen = torch.Generator(device="cuda").manual_seed(0)
    inp = torch.rand((B, C, H + 4, W + 4), device="cuda", generator=gen)
    w = torch.zeros((B, F * F, H, W), device="cuda")
    w[:, 12] = 1.0
    z = torch.zeros_like(w)
    out = adacof.adacof_forward(inp, w, z, z, d)
    assert torch.equal(out, inp[:, :, 2:-2, 2:-2])
    del z
    w = torch.softmax(torch.randn((B, F * F, H, W), device="cuda", generator=gen), 1)
    oi = (3 * torch.randn((B, F * F, H, W), device="cuda", generator=gen)).clamp_(-16, 16)
    oj = (3 * torch.randn((B, F * F, H, W), device="cuda", generator=gen)).clamp_(-16, 16)
    inp2 = torch.rand((B, C, H + 4, W + 4), device="cuda", generator=gen)
    o1 = adacof.adacof_forward(inp, w, oi, oj, d)
    o2 = adacof.adacof_forward(inp2, w, oi, oj, d)
    o12 = adacof.adacof_forward(inp + 2 * inp2, w, oi, oj, d)
    assert float((o12 - (o1 + 2 * o2)).abs().max()) < 2e-5
    # slab vs oracle: rows 500..515 of sample 3
    r0, r1 = 500, 516
    sl = lambda t: t[3:4, :, r0:r1].contiguous().cpu().numpy()
    ref = oa.forward(inp[3:4, :, r0:r1 + 4].contiguous().cpu().numpy(), sl(w), sl(oi), sl(oj), d)
    # the slab oracle clamps rows at the slab edge; rows whose taps may leave the slab are excluded by
    # comparing only pixels whose row offsets stay inside (|off|<=16 can leave a 20-row slab) -> compare
    # on a version with row offsets zeroed instead
    oi0 = torch.zeros_like(oi[3:4])
    o_full = adacof.adacof_forward(inp[3:4].contiguous(), w[3:4].contiguous(), oi0, oj[3:4].contiguous(), d)
    ref = oa.forward(inp[3:4, :, r0:r1 + 4].contiguous().cpu().numpy(), sl(w), np.zeros_like(sl(oi)), sl(oj), d)
    assert np.abs(o_full[:, :, r0:r1].cpu().numpy() - ref).max() <= TOL_FWD
