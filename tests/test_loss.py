"""fvfi.loss (drop-in for src/train/loss.py, the PhaseNet training loss): known-answer values on CPU tensors (the loss itself is
plain tensor arithmetic; the image term's backward through the pyramid is covered by tests/test_pyramid_gpu.py /
test_models_gpu.py::test_phasenet_training_step)."""
import math
import types

import torch

from collections import namedtuple

V = namedtuple("values", "high_level, phase, amplitude, low_level")


def _case(seed, P=3, nb=4, sizes=((16, 20), (11, 14), (8, 10))):
    g = torch.Generator().manual_seed(seed)
    ph_o = [(torch.rand((P * nb, 1, h, w), generator=g) * 2 - 1) * math.pi for h, w in sizes]
    ph_t = [(torch.rand((P * nb, 1, h, w), generator=g) * 2 - 1) * math.pi for h, w in sizes]
    out, tgt = torch.rand((P, 32, 40), generator=g), torch.rand((P, 32, 40), generator=g)
    mk = lambda ph: V(high_level=None, phase=ph, amplitude=[None] * len(ph), low_level=None)
    return mk(ph_o), mk(ph_t), out, tgt


def test_get_loss_known_answers():
    """No reference needed: identical pyramids -> pure L1; a constant phase offset d on every coefficient -> L1 + 0.005 * levels * nb * |wrap(d)|
    (one mean per level and orientation, summed: loss.py:10-16), including offsets beyond pi that wrap."""
    from fvfi.loss import get_loss, wrapped_phase_l1
    pyr = types.SimpleNamespace(nbands=4)
    vo, _, out, tgt = _case(3)
    l1 = float(torch.nn.functional.l1_loss(out, tgt))
    total, p1, p2 = get_loss(vo, vo, out, tgt, pyr)
    assert abs(float(total) - l1) <= 1e-7 and abs(float(p1) - 100.0) <= 1e-4 and abs(float(p2)) <= 1e-6
    for d in (0.3, -2.0, 4.0, 2 * math.pi + 0.25):
        wrapped = abs(math.atan2(math.sin(d), math.cos(d)))
        vt = vo._replace(phase=[p + d for p in vo.phase])
        total, p1, p2 = get_loss(vo, vt, out, tgt, pyr)
        want = l1 + 0.005 * len(vo.phase) * 4 * wrapped
        assert abs(float(total) - want) <= 2e-6 * max(1.0, want), d
        assert abs(float(p1) + float(p2) - 100.0) <= 1e-3
    x = torch.tensor([0.0, 3.0, -3.0])
    y = torch.tensor([0.5, -3.0, 3.0])                       # 3 -> -3 is a step of 2*pi - 6 = 0.283, not 6
    assert abs(float(wrapped_phase_l1(x, y)) - (0.5 + 2 * (2 * math.pi - 6)) / 3) <= 1e-6
    # levels given as the int 0 (not predicted, phase_net.py:91-93) are skipped
    vz = vo._replace(phase=[vo.phase[0], 0, vo.phase[2]])
    total, _, _ = get_loss(vz, vo, out, tgt, pyr)
    assert abs(float(total) - l1) <= 1e-7
