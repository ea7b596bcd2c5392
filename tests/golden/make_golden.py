"""Generate golden vectors by running the UNMODIFIED reference (a checkout of
CGCL-codes/DorPatch @ 0751fd4) under the CPU shim of oracle/ref_shim.py.  The resulting .npz
fixture is committed next to this script, so the test suite never needs the reference.

    python tests/golden/make_golden.py --reference <path of the reference checkout>

Pins (SURVEY.md section 4): G1 mask geometry, G2 utils.clip, G3 losses + gradients,
G4 patch_selection, G5/G6 generate trajectories (tiny stand-in classifier: targeted 10 steps,
and untargeted 1100 steps crossing the i==500 targeted switch, the i>=1000 failed-set sampling
and the lr-decay path), G7 PatchCleanser records, G9 a ResNetV2-50 trajectory at 112 px,
G10 a 25-step targeted dropout-2 trajectory (tiny classifier, absolute target label).
The G2 inputs are not stored: g2_inputs() re-draws them from their seed.
"""
import contextlib
import io
import os
import random
import shutil
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import ref_shim, resnetv2 as OR  # noqa: E402


class TinyNet(torch.nn.Module):
    """Deterministic stand-in classifier for control-flow pins (x in [0,1] -> 1000 logits)."""

    def __init__(self, seed=0, classes=1000):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.w1 = torch.nn.Parameter(torch.randn(8, 3, 3, 3, generator=g) * 0.5)
        self.w2 = torch.nn.Parameter(torch.randn(16, 8, 3, 3, generator=g) * 0.3)
        self.fc = torch.nn.Parameter(torch.randn(classes, 16, generator=g) * 2.0)

    def forward(self, x):
        h = torch.relu(torch.nn.functional.conv2d(x - 0.5, self.w1, stride=2, padding=1))
        h = torch.relu(torch.nn.functional.conv2d(h, self.w2, stride=2, padding=1))
        return h.mean((2, 3)) @ self.fc.t()


def seed_all(s=1234):
    random.seed(s)
    torch.manual_seed(s)
    np.random.seed(s)


def g2_inputs():
    """The seeded inputs of G2 (image, mask, pattern, output weights) and the generator, which G3 and G4 draw on from there."""
    g = torch.Generator().manual_seed(11)
    x = torch.rand(3, 3, 56, 56, generator=g)
    m = torch.rand(3, 1, 56, 56, generator=g)
    p = torch.rand(3, 3, 56, 56, generator=g)
    m[1] *= 0.01
    w = torch.rand(3, 3, 56, 56, generator=g)
    return g, x, m, p, w


G10_KW = dict(patch_budget=0.12, n_classes=1000, targeted=True, y=torch.tensor([7]), max_iterations=25, sampling_size=3,
              dropout=2)


def g10_input():
    return torch.rand(1, 3, 56, 56, generator=torch.Generator().manual_seed(21))


def run_generate(ref, net, x, **kw):
    """Reference generate in a scratch cwd (it writes stage-0 artefacts relative to cwd)."""
    cwd = os.getcwd()
    tmp = tempfile.mkdtemp()
    os.chdir(tmp)
    try:
        os.makedirs("r/sub")
        buf = io.StringIO()
        seed_all()
        with contextlib.redirect_stdout(buf):
            m, p = ref.attack.DorPatch().generate(net, x, save_dir="r/sub", batch_id=0, **kw)
        log = [l for l in buf.getvalue().splitlines() if not l.startswith("mask size")]
        rng_np = np.random.get_state()[1][:4].copy()
        rng_t = torch.rand(3).numpy()
        return m.detach().numpy(), p.detach().numpy(), log, rng_np, rng_t
    finally:
        os.chdir(cwd)
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="checkout of the unmodified reference (CGCL-codes/DorPatch @ 0751fd4)")
    root = os.path.abspath(ap.parse_args().reference)
    assert ref_shim.available(root), "no reference at %s" % root
    torch.set_num_threads(8)
    out = {}
    with ref_shim.reference_modules(root) as ref:
        A, U, PC = ref.attack, ref.utils, ref.PatchCleanser
        # ---- G1 geometry -----------------------------------------------------------------
        with contextlib.redirect_stdout(io.StringIO()):
            for H in (56, 224):
                for r in (0.015, 0.03, 0.06, 0.12):
                    mw = PC.MaskWindow(H, r, 1)
                    out["g1_geom_%d_%s" % (H, r)] = np.array([mw.mask_size, mw.stride, mw.window_size])
                    out["g1_single_%d_%s" % (H, r)] = np.packbits(mw.mask_set.numpy())
                    dm = mw.double_mask_set.numpy()
                    out["g1_double_sum_%d_%s" % (H, r)] = dm.reshape(dm.shape[0], -1).sum(1).astype(np.int32)
                    out["g1_double_probe_%d_%s" % (H, r)] = np.packbits(dm[[0, 1, 35, 36, 300, 629]])
        # ---- G2 clip -----------------------------------------------------------------------
        g, x, m, p, w = g2_inputs()
        mm, pp = m.clone().requires_grad_(True), p.clone().requires_grad_(True)
        d = U.clip(mm, pp, x, 4.0)
        (d * w).sum().backward()
        out.update(g2_delta=d.detach().numpy(), g2_gm=mm.grad.numpy(), g2_gp=pp.grad.numpy())
        # ---- G3 losses + gradients ------------------------------------------------------------
        xa = torch.rand(2, 3, 56, 56, generator=g).requires_grad_(True)
        lv, lr_, ud = A.local_variance(xa)
        mv = A.min_var_weighted_variance(xa)
        lvx = A.local_variance(x[:2])[0].mean(1)
        ls = torch.mean(mv.mean(1) / (lvx + 1e-5), (1, 2))
        ls.sum().backward()
        out.update(g3_x=xa.detach().numpy(), g3_lv=lv.detach().numpy(), g3_mv=mv.detach().numpy(),
                   g3_ls=ls.detach().numpy(), g3_ls_grad=xa.grad.numpy())
        ma = torch.rand(2, 1, 56, 56, generator=g)
        ma[0, 0, :7, 7:14] = 0
        ma = ma.requires_grad_(True)
        cg = torch.nn.Conv2d(1, 1, 7, stride=7, bias=False)
        cg.weight.data[:] = 1
        cd = torch.nn.Conv2d(1, 1, 7, stride=7, bias=False)   # window = 56 // 8 = 7
        cd.weight.data[:] = 1
        den = cd(ma).view((2, -1)).var(1)
        gl = 7 * cg(ma ** 2).sqrt().sum((1, 2, 3))
        (den * 1e-3 + gl * 1e-5).sum().backward()
        out.update(g3_mask=ma.detach().numpy(), g3_density=den.detach().numpy(), g3_lasso=gl.detach().numpy(),
                   g3_mask_grad=ma.grad.numpy())
        lg = torch.randn(6, 1000, generator=g)
        yy = torch.tensor([1, 5, 999, 0, 17, 400])
        lg[3, 0] = 50.0
        for tg in (False, True):
            l2 = lg.clone().requires_grad_(True)
            v = A.CW_loss(1000, tg, 0.1)(l2, yy)
            v.sum().backward()
            out["g3_cw_%d" % tg] = v.detach().numpy()
            out["g3_cw_grad_%d" % tg] = l2.grad.numpy()
        out["g3_cw_logits"], out["g3_cw_y"] = lg.numpy(), yy.numpy()
        # ---- G4 patch_selection -------------------------------------------------------------------
        mk = torch.rand(2, 1, 56, 56, generator=g)
        mk[1, 0, :28] = 0
        for bud in (0.05, 0.10, 0.12, 0.9):
            with torch.no_grad():
                out["g4_sel_%s" % bud] = np.packbits(A.DorPatch().patch_selection(mk, bud).numpy().astype(bool))
        out["g4_mask"] = mk.numpy()
        # ---- G5/G6 trajectories with the tiny classifier ---------------------------------------------
        tiny = TinyNet().eval()
        xs = torch.rand(1, 3, 56, 56, generator=torch.Generator().manual_seed(5))
        with torch.no_grad():
            y0 = tiny(xs).argmax(-1)
        runs = {
            "t10": dict(patch_budget=0.12, n_classes=1000, targeted=True, y=(y0 + 3) % 1000, max_iterations=10,
                        sampling_size=1, dropout=1),
            "u1100": dict(patch_budget=0.10, n_classes=1000, targeted=False, max_iterations=1100, sampling_size=6,
                          dropout=2),
            "t300dual": dict(patch_budget=0.05, n_classes=1000, targeted=True, y=(y0 + 9) % 1000,
                             max_iterations=300, sampling_size=4, dropout=1, dual=True, lr=0.05),
        }
        for name, kw in runs.items():
            mo, po, log, rn, rt = run_generate(ref, tiny, xs, **kw)
            out["g6_%s_mask" % name] = np.packbits(mo.astype(bool)) if set(np.unique(mo)) <= {0.0, 1.0} else mo
            out["g6_%s_pattern" % name] = po
            out["g6_%s_log" % name] = np.array(log)
            out["g6_%s_rng_np" % name] = rn
            out["g6_%s_rng_t" % name] = rt
            print(name, "log lines", len(log), "mask mean", mo.mean())
        out["g6_x"] = xs.numpy()
        # ---- G7 PatchCleanser records -------------------------------------------------------------------
        with contextlib.redirect_stdout(io.StringIO()):
            for r in (0.03, 0.12):
                d = PC.PatchCleanser(PC.MaskWindow(56, r, 1), tiny)
                for k in range(3):
                    img = torch.rand(3, 56, 56, generator=torch.Generator().manual_seed(100 + k))
                    with torch.no_grad():
                        rec = d.robust_predict(img, True)
                    out["g7_%s_%d_pred" % (r, k)] = np.array([rec.prediction, int(rec.certification)])
                    out["g7_%s_%d_p1" % (r, k)] = rec.preds_1
                    out["g7_%s_%d_p2" % (r, k)] = rec.preds_2.astype(np.int64)
        # ---- G9 ResNetV2-50 trajectory at 112 px (BASELINE config 1 shape: 1 image, few-step PGD) ---------
        params = OR.random_init(seed=0, affine_jitter=0.1)
        net = OR.OracleNet(params).eval()
        xr = torch.rand(1, 3, 112, 112, generator=torch.Generator().manual_seed(7))
        with torch.no_grad():
            yr = net(xr).argmax(-1)
        kw = dict(patch_budget=0.12, n_classes=1000, targeted=True, y=(yr + 17) % 1000, max_iterations=6,
                  sampling_size=4, dropout=1)
        mo, po, log, rn, rt = run_generate(ref, net, xr, **kw)
        out["g9_mask"] = np.packbits(mo.astype(bool))
        out["g9_pattern"] = po.astype(np.float16)
        out["g9_log"] = np.array(log)
        out["g9_rng_np"] = rn
        out["g9_target"] = ((yr + 17) % 1000).numpy()
        # ---- G10 a dropout-2 trajectory with an absolute target label (tiny classifier) ----------------------------
        mo, po, log, rn, rt = run_generate(ref, tiny, g10_input(), **G10_KW)
        out.update(g10_mask=mo, g10_pattern=po, g10_log=np.array(log), g10_rng_np=rn)
    np.savez_compressed(os.path.join(HERE, "reference_golden.npz"), **out)
    print("wrote", os.path.join(HERE, "reference_golden.npz"), os.path.getsize(os.path.join(HERE, "reference_golden.npz")))


if __name__ == "__main__":
    main()
