"""CPU tests: the oracle restatements of the networks / fusion recipe (oracle/nets.py,
oracle/fusion_pipeline.py) against the committed golden fixtures produced by the REAL reference
modules (tests/golden/make_golden_models.py, make_golden_r2.py)."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import fusion_pipeline as fp


def _fixtures(golden_dir):
    return sorted(glob.glob(os.path.join(golden_dir, "pipeline_ref_*.npz")))


def test_pipeline_oracle_matches_reference_golden(golden_dir):
    f = os.path.join(golden_dir, "pipeline_ref_B1_64x64_s0.npz")  # 64x64, B=1 (a few seconds on CPU)
    z = np.load(f)
    B, H, W, seed = [int(v) for v in z["meta"]]
    state = fp.seeded_state(seed)
    chk = [float(sum(v.double().sum() for v in state[n].values())) for n in ("phase_net", "fusion_net", "adacof")]
    assert np.allclose(chk, z["checksum"], rtol=1e-9), "seeded init differs from the fixture's"
    rgb1, rgb2 = fp.seeded_frames(B, H, W, seed)
    st = {}
    fp.interp(fp.oracle_backend(state, hw=(H, W), threads=4), rgb1, rgb2, st)
    for k in ("lab1", "ada_pred", "flow_var_map", "lab_pred", "phase_pred", "phase_uncertainty", "ada_uncertainty",
              "base", "final"):
        assert np.abs(st[k].numpy() - z[k]).max() <= 2e-6, k


def test_oracle_nets_equal_reference_modules(golden_dir):
    """Every stage of the recipe, batch 2, against the stored outputs of the reference's own modules (images stored
    subsampled by ``<k>__stride``)."""
    z = np.load(os.path.join(golden_dir, "pipeline_ref_B2_64x96_s1.npz"))
    B, H, W, seed = [int(v) for v in z["meta"]]
    state = fp.seeded_state(seed)
    chk = [float(sum(v.double().sum() for v in state[n].values())) for n in ("phase_net", "fusion_net", "adacof")]
    assert np.allclose(chk, z["checksum"], rtol=1e-9), "seeded init differs from the fixture's"
    rgb1, rgb2 = fp.seeded_frames(B, H, W, seed)
    b = {}
    fp.interp(fp.oracle_backend(state, hw=(H, W), threads=4), rgb1, rgb2, b)
    assert len(b) == 12
    for k in b:
        sl = int(z[k + "__stride"]) if k + "__stride" in z.files else 1
        assert np.abs(b[k].numpy()[..., ::sl, ::sl] - z[k]).max() <= 1e-6, k


def test_phasenet256_oracle_matches_reference_golden_and_fp64_budget(golden_dir):
    """configs[0] fixture: the oracle restatement (fp32) reproduces the reference modules' outputs, and its fp64 mode reproduces
    the stored arbiter (so the budgets the GPU tests use are what the fixture says)."""
    z = np.load(os.path.join(golden_dir, "phasenet_ref_256x256_s5.npz"))
    B, H, W, seed = [int(v) for v in z["meta"]]
    state = fp.seeded_state(seed)
    rgb1, rgb2 = fp.seeded_frames(B, H, W, seed)
    st32, st64 = {}, {}
    fp.interp_phasenet(fp.oracle_backend(state, hw=(H, W), threads=4), rgb1, rgb2, st32)
    fp.interp_phasenet(fp.oracle_backend(state, hw=(H, W), threads=4, precision="fp64"), rgb1, rgb2, st64)
    for k in ("lab_pred", "phase_pred", "low_level", "amp3", "amp9"):
        sl = int(z[k + "__stride"]) if k + "__stride" in z.files else 1
        a32 = st32[k].numpy()[..., ::sl, ::sl]
        a64 = st64[k].numpy()[..., ::sl, ::sl]
        assert np.abs(a32 - z[k]).max() <= 2e-6, k
        f64 = z[k].astype(np.float64) - z[k + "__d64"].astype(np.float64) / 1e4
        assert np.abs(a64 - f64).max() <= 2e-3 * float(z[k + "__budget"]) + 1e-7, k      # float16 storage of the difference
        assert float(np.abs(st32[k].numpy() - st64[k].numpy()).max()) == pytest.approx(float(z[k + "__budget"]), rel=1e-3, abs=1e-9)


def test_reference_recipe_is_discontinuous_at_the_phase_wrap():
    """Why the parity runs align the +-pi branch (tests/_parity.py: WrapAligner).  On the CPU restatement of the reference (pinned
    equal to the reference's own modules): perturb the decomposition of a 256x256 pair by white noise of 5e-7 of each level's
    maximum -- the size of fp32 FFT rounding, i.e. what ANY other FFT build does to it.  A handful of the 2.6 M coefficients sit so
    close to the negative real axis that their wrapped phase imag(log z) (src/train/pyramid.py:63) jumps between +pi and -pi, and
    those few jumps alone move PhaseNet's output by ~1e-4 (with the shipped phase_net.pt: ~4e-3); with the jumps undone the same
    perturbation moves it by ~3e-7."""
    H = W = 256
    state = fp.seeded_state(4)
    rgb1, rgb2 = fp.seeded_frames(1, H, W, 4)
    be = fp.oracle_backend(state, hw=(H, W), threads=4)
    lab1, lab2 = fp.rgb2lab_planes(rgb1), fp.rgb2lab_planes(rgb2)
    vals = be.pyr.filter(torch.cat((lab1.reshape(-1, H, W), lab2.reshape(-1, H, W)), 0))

    def run(v):
        vin = be.phase_net.normalize_vals(be.get_concat_layers_inf(be.pyr, be.separate_vals(v, 2)))
        with torch.no_grad():
            return be.pyr.inv_filter(be.phase_net(vin))
    base = run(vals)
    g = torch.Generator().manual_seed(0)
    ph, am, ph_undone, flips = [], [], [], 0
    for p, a in zip(vals.phase, vals.amplitude):
        z = a.double() * torch.exp(1j * p.double())
        noise = torch.randn(z.shape, generator=g, dtype=torch.float64) + 1j * torch.randn(z.shape, generator=g, dtype=torch.float64)
        z = z + noise * (5e-7 * float(a.max()) / 3)
        pn, an = torch.angle(z).float(), z.abs().float()
        fl = (pn - p).abs() > 3.0
        flips += int(fl.sum())
        ph.append(pn)
        am.append(an)
        ph_undone.append(torch.where(fl, p, pn))
    with_flips = float((run(vals._replace(phase=ph, amplitude=am)) - base).abs().max())
    undone = float((run(vals._replace(phase=ph_undone, amplitude=am)) - base).abs().max())
    print("flips %d, output change with flips %.2e, with the flips undone %.2e" % (flips, with_flips, undone))
    assert 1 <= flips <= 20
    assert undone <= 2e-6
    assert with_flips >= 20 * undone and with_flips >= 2e-5


def test_synth_generators_equal_oracle_generators():
    """fvfi.synth (what bench.py / tools use for seeded weights and frames) == the oracle's generators (what the fixtures use)."""
    from fvfi import synth
    a, b = fp.seeded_state(3), synth.seeded_state(3)
    for k in a:
        assert list(a[k].keys()) == list(b[k].keys())
        assert all(torch.equal(a[k][n], b[k][n]) for n in a[k])
    assert all(torch.equal(p, q) for p, q in zip(fp.seeded_frames(2, 64, 96, 1), synth.seeded_frames(2, 64, 96, 1)))


def test_lab_round_trip_and_known_values():
    from oracle import lab
    rgb = np.random.default_rng(0).random((5, 7, 3))
    assert np.abs(lab.lab2rgb(lab.rgb2lab(rgb)) - rgb).max() < 1e-6
    # white, black, mid-grey (CIE L* of sRGB 0.5 is 53.389)
    assert np.allclose(lab.rgb2lab(np.ones((1, 1, 3)))[0, 0], [100, 0, 0], atol=2e-2)
    assert np.allclose(lab.rgb2lab(np.zeros((1, 1, 3)))[0, 0], [0, 0, 0], atol=1e-9)
    assert abs(lab.rgb2lab(np.full((1, 1, 3), 0.5))[0, 0, 0] - 53.389) < 1e-2


def test_lab_oracle_agrees_with_opencv():
    """Coarse, independent anchor for the UNPINNED Lab oracle (scikit-image, what the reference calls in src/train/transform.py:6-49,
    is not installed): OpenCV's float RGB<->Lab implements the same standard (sRGB companding, D65, CIE 1976) with table-interpolated
    gamma / cube root, so it agrees only to a few tenths of a Lab unit -- enough to catch a wrong white point, matrix or threshold
    (each of which moves values by > 1 unit), not enough to pin the last digits."""
    cv2 = pytest.importorskip("cv2")
    from oracle import lab
    rng = np.random.default_rng(0)
    rgb = rng.random((96, 80, 3)).astype(np.float32)
    rgb[:8] *= 0.02                                        # the linear segment of the sRGB curve and of f(t)
    ours = lab.rgb2lab(rgb)
    theirs = cv2.cvtColor(rgb, cv2.COLOR_RGB2Lab).astype(np.float64)
    assert float(np.abs(ours - theirs).max()) <= 0.5, float(np.abs(ours - theirs).max())
    back = cv2.cvtColor(theirs.astype(np.float32), cv2.COLOR_Lab2RGB).astype(np.float64)
    assert float(np.abs(lab.lab2rgb(theirs) - back).max()) <= 2e-3
