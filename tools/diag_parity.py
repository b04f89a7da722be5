"""Error breakdown of the PhaseNet branch (developer tool, GPU box): which stage carries the difference to the CPU oracle?
    python tools/diag_parity.py H W [ckpt]
A  GPU decomposition vs oracle fp32 / fp64 (complex coefficients, relative to the level maximum)
B  GPU PhaseNet on the ORACLE's decomposition vs the oracle's PhaseNet (per conv back end / operand split)
C  GPU reconstruction of the ORACLE's predicted values vs the oracle's inv_filter
D  the whole branch on the GPU vs oracle fp32 / fp64
"""
import os, sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "fusion-method-for-video-frame-interpolation_b200")]
from oracle import fusion_pipeline as fp, nets
from fvfi import conv as tc, utils
from fvfi.pipeline import FusionPipeline
from fvfi.pyramid import DecompValues

H, W = int(sys.argv[1]), int(sys.argv[2])
ckpt = len(sys.argv) > 3 and sys.argv[3] == "ckpt"
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
state = fp.seeded_state(4)
if ckpt:
    state["phase_net"] = torch.load(os.path.join(ROOT, "oracle/_ref/phase_net.pt"), map_location="cpu")
rgb1, rgb2 = fp.seeded_frames(1, H, W, 4)
torch.set_num_threads(os.cpu_count())


def cplx(ph, am):
    return am.double() * torch.exp(1j * ph.double())


def oracle_branch(prec):
    be = fp.oracle_backend(state, hw=(H, W), threads=8, precision=prec)
    dt = be.dtype
    lab1, lab2 = fp.rgb2lab_planes(rgb1.to(dt), dt), fp.rgb2lab_planes(rgb2.to(dt), dt)
    img = torch.cat((lab1.reshape(-1, H, W), lab2.reshape(-1, H, W)), 0)
    vals = be.pyr.filter(img)
    vin = be.phase_net.normalize_vals(be.get_concat_layers_inf(be.pyr, be.separate_vals(vals, 2)))
    with torch.no_grad():
        pred = be.phase_net(vin)
    rec = be.pyr.inv_filter(pred)
    return dict(img=img, vals=vals, pred=pred, rec=rec, be=be)


o32, o64 = oracle_branch("fp32"), oracle_branch("fp64")
pipe = FusionPipeline(H, W, "cuda")
pipe.load_state(state)
pyr = pipe.pyr
L = pyr.height - 2
img = o32["img"].float().cuda()
with torch.no_grad():
    # ---- A
    gv = pyr.filter(img)
    print("A  decomposition: max |coef_gpu - coef_oracle| / max|level|  (vs fp32 | vs fp64 | oracle fp32 vs fp64)")
    for l in range(L):
        g = cplx(gv.phase[l].cpu(), gv.amplitude[l].cpu())
        a, b = cplx(o32["vals"].phase[l], o32["vals"].amplitude[l]), cplx(o64["vals"].phase[l], o64["vals"].amplitude[l])
        m = float(b.abs().max())
        print("   level %2d %4dx%-4d  %.2e | %.2e | %.2e" % (l, g.shape[-2], g.shape[-1], float((g - a).abs().max()) / m,
                                                             float((g - b).abs().max()) / m, float((a - b).abs().max()) / m))
    print("   low  %.2e | %.2e | %.2e" % tuple(float((x.double() - y.double()).abs().max()) for x, y in
                                              ((gv.low_level.cpu(), o32["vals"].low_level), (gv.low_level.cpu(), o64["vals"].low_level),
                                               (o32["vals"].low_level, o64["vals"].low_level))))
    # ---- B: GPU network on the oracle's (fp32) decomposition
    ov = o32["vals"]
    dv = DecompValues(high_level=ov.high_level.cuda(), low_level=ov.low_level.cuda(), phase=[p.cuda() for p in ov.phase],
                      amplitude=[a.cuda() for a in ov.amplitude])

    def run_net():
        vin = pipe.phase_net.normalize_vals(utils.get_concat_layers_inf(pyr, utils.separate_vals(dv, 2)))
        return pipe.phase_net(vin)
    print("B  PhaseNet on the oracle's decomposition: max |coef - oracle fp32 coef| / max|level| per level, then low_level abs")
    for name in ("f16x3", "tf32x3", "cudnn"):
        if name != "cudnn":
            with tc.forced_precision(name):
                gp = run_net()
        else:
            with torch.enable_grad():              # PhaseNet's differentiable graph = torch convolutions (cuDNN fp32)
                gp = run_net()
            gp = gp._replace(phase=[p.detach() for p in gp.phase], amplitude=[a.detach() for a in gp.amplitude], low_level=gp.low_level.detach())
        errs = []
        for l in range(L):
            g = cplx(gp.phase[l].cpu(), gp.amplitude[l].cpu())
            a = cplx(o32["pred"].phase[l], o32["pred"].amplitude[l])
            errs.append(float((g - a).abs().max()) / float(a.abs().max()))
        ref64 = [float((cplx(o32["pred"].phase[l], o32["pred"].amplitude[l]) - cplx(o64["pred"].phase[l], o64["pred"].amplitude[l])).abs().max())
                 / float(cplx(o64["pred"].phase[l], o64["pred"].amplitude[l]).abs().max()) for l in range(L)]
        print("   %-7s" % name, " ".join("%.1e" % e for e in errs), "| low %.2e" % float((gp.low_level.cpu() - o32["pred"].low_level).abs().max()))
    print("   (oracle fp32 vs fp64, own inputs)", " ".join("%.1e" % e for e in ref64),
          "| low %.2e" % float((o32["pred"].low_level.double() - o64["pred"].low_level).abs().max()))
    # ---- C: GPU reconstruction of the oracle's predicted values
    op = o32["pred"]
    pv = DecompValues(high_level=op.high_level.cuda(), low_level=op.low_level.cuda(), phase=[p.cuda() for p in op.phase],
                      amplitude=[a.cuda() for a in op.amplitude])
    rec = pyr.inv_filter(pv).cpu()
    print("C  reconstruction of the oracle's prediction: max abs vs oracle fp32 %.2e ; oracle fp32 vs fp64 (own values) %.2e"
          % (float((rec - o32["rec"]).abs().max()), float((o32["rec"].double() - o64["rec"]).abs().max())))
    # ---- D: whole branch
    pipe.stages = {}
    pipe.phase_interp(rgb1.cuda(), rgb2.cuda())
    lp = pipe.stages["lab_pred"].reshape(-1, H, W).cpu()
    print("D  whole branch: lab_pred max abs vs oracle fp32 %.2e, vs fp64 %.2e ; oracle fp32 vs fp64 %.2e"
          % (float((lp - o32["rec"]).abs().max()), float((lp.double() - o64["rec"]).abs().max()),
             float((o32["rec"].double() - o64["rec"]).abs().max())))
    pipe.stages = None
