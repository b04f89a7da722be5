"""Drop-in for the DecompValues plumbing of the reference's ``src/train/utils.py`` (only the
functions on the fusion path; same names, argument meaning and return layouts)."""
import math

import torch

from .pyramid import DecompValues


def get_concat_layers_inf(pyr, vals_list):
    """utils.py:47-80.  [P*nb,1,h,w] per frame -> [P, nb*num_img, h, w], lists reversed to COARSEST first."""
    nbands, height = pyr.nbands, pyr.height
    high_level = torch.cat([e.high_level for e in vals_list], 1)
    low_level = torch.cat([e.low_level for e in vals_list], 1)
    rs = lambda x: x.reshape(x.shape[0] // nbands, nbands, x.shape[2], x.shape[3])
    phase = [torch.cat([rs(e.phase[i]) for e in vals_list], 1) for i in range(height - 2)]
    amplitude = [torch.cat([rs(e.amplitude[i]) for e in vals_list], 1) for i in range(height - 2)]
    return DecompValues(high_level=high_level, low_level=low_level, phase=phase[::-1], amplitude=amplitude[::-1])


def get_concat_layers(pyr, vals1, vals2):
    """utils.py:19-44."""
    return get_concat_layers_inf(pyr, [vals1, vals2])


def separate_vals(vals, num_input):
    """utils.py:83-127.  Splits the batch dimension into ``num_input`` per-frame DecompValues (views)."""
    def split(t):
        return None if t is None else t.reshape(num_input, -1, t.shape[2], t.shape[3])   # None: level not computed
    low, high = split(vals.low_level), split(vals.high_level)
    ph = [split(p) for p in vals.phase]
    am = [split(a) for a in vals.amplitude]
    out = []
    for i in range(num_input):
        out.append(DecompValues(high_level=high[i].unsqueeze(1), low_level=low[i].unsqueeze(1),
                                phase=[None if p is None else p[i].unsqueeze(1) for p in ph],
                                amplitude=[None if a is None else a[i].unsqueeze(1) for a in am]))
    return out


def pair_vals(vals, q, nbands):
    """The two per-frame DecompValues of a decomposition in which frame 2 of pair-plane p is plane p + q (views): frame 1 = planes
    [0, P), frame 2 = planes [q, q + P), P = N - q.  q = N / 2 is ``separate_vals(vals, 2)``; q = 3 is a clip of consecutive
    frames decomposed once (pair t = frames t, t + 1)."""
    N = vals.low_level.shape[0]
    P = N - q
    planes = lambda t, k: t[k:k + P]
    bands = lambda t, k: None if t is None else t[k * nbands:(k + P) * nbands]
    return [DecompValues(high_level=planes(vals.high_level, k), low_level=planes(vals.low_level, k),
                         phase=[bands(p, k) for p in vals.phase], amplitude=[bands(a, k) for a in vals.amplitude])
            for k in (0, q)]


def combine_values(vals_list):
    """utils.py:208-240."""
    return DecompValues(
        high_level=torch.cat([v.high_level for v in vals_list], 0),
        low_level=torch.cat([v.low_level for v in vals_list], 0),
        phase=[torch.cat([v.phase[i] for v in vals_list], 0) for i in range(len(vals_list[0].phase))],
        amplitude=[torch.cat([v.amplitude[i] for v in vals_list], 0) for i in range(len(vals_list[0].phase))])


def get_last_value_levels(vals, use_levels=1):
    """utils.py:242-280: keep high_level and the first ``use_levels`` (finest) band levels, zero the rest."""
    z = torch.zeros_like
    return DecompValues(high_level=vals.high_level.clone(), low_level=z(vals.low_level),
                        phase=[p.clone() if i < use_levels else z(p) for i, p in enumerate(vals.phase)],
                        amplitude=[a.clone() if i < use_levels else z(a) for i, a in enumerate(vals.amplitude)])


def get_first_value_levels(vals, use_levels=1):
    """utils.py:282-320: keep low_level and the last ``use_levels`` (coarsest) band levels, zero the rest."""
    z = torch.zeros_like
    n = len(vals.phase)
    return DecompValues(high_level=z(vals.high_level), low_level=vals.low_level.clone(),
                        phase=[z(p) if i < n - use_levels else p.clone() for i, p in enumerate(vals.phase)],
                        amplitude=[z(a) if i < n - use_levels else a.clone() for i, a in enumerate(vals.amplitude)])


def subtract_values(vals1, vals2):
    """utils.py:322-346: element-wise |a-b| of every component."""
    return DecompValues(high_level=(vals1.high_level - vals2.high_level).abs(),
                        low_level=(vals1.low_level - vals2.low_level).abs(),
                        phase=[(a - b).abs() for a, b in zip(vals1.phase, vals2.phase)],
                        amplitude=[(a - b).abs() for a, b in zip(vals1.amplitude, vals2.amplitude)])


def exchange_vals(val_base, val_changer, start, end):
    """utils.py:145-152."""
    for level in range(start, end):
        val_base.phase[level] = val_changer.phase[level]
        val_base.amplitude[level] = val_changer.amplitude[level]
    return val_base


def calc_pyr_height(img):
    """utils.py:168-171."""
    size = img.shape[1:]
    return int(math.ceil((math.log2(min(size)) - 3) * 2) + 2)


def pad_img_size(h, w):
    """Target square size of utils.py:155-165 (pad to a power of sqrt(2)): 1080p -> 2048."""
    p = lambda s: int(2 ** (math.ceil(math.log2(s) * 2) / 2))
    return max(p(h), p(w))
