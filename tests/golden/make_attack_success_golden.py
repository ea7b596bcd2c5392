"""Freeze the END METRIC of the reference pipeline (main.py:128-187) on the CPU oracle:
generate -> paste -> PatchCleanser at the four ratios, per image, for K synthetic images.

    python tests/golden/make_attack_success_golden.py [--K 16 --iters 200 --S 8]                       -> attack_success_golden.npz
    python tests/golden/make_attack_success_golden.py --perturb 1e-7 --save-adv 0 --out attack_success_noise.npz      (noise floor)
    python tests/golden/make_attack_success_golden.py --eps 16 --save-adv 0 --out attack_success_saturated.npz   (saturated regime)

The oracle (oracle/attack.py, oracle/patchcleanser.py) is pinned bit-exactly to the unmodified
reference (tests/test_oracle_golden.py, tests/test_oracle_vs_reference.py), so its success /
certification bits ARE the reference's on these seeds.  Protocol per image i (a B == 1 run, the
only batch size the reference supports): seed python / torch / numpy with SEED0 + i
(utils.set_random_seed), x_i = rand(3,112,112) from a generator seeded IMG_SEED0 + i,
untargeted DorPatch.generate(patch_budget 0.12, dropout 1, sampling_size S, max_iterations iters,
eps 4), adv_x = x + clip(mask, pattern, x, eps) (main.py:140-141), robust_predict(adv_x, certify)
for ratios 0.015/0.03/0.06/0.12 (main.py:61,151), model(adv_x).argmax (main.py:156).
tests/test_gpu_attack_success.py replays the same protocol on the native engine (fp32 / tf32 /
bf16) and compares the bits and the main.py:162-185 rates.  Output: attack_success_golden.npz.
The final adversarial images are stored as adv_delta = adv_x - x_i (x_i unperturbed), which is
mostly zero and compresses; image(i) + adv_delta[i] reproduces adv_x bit for bit (asserted).
"""
import os
import random
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import attack as OA, patchcleanser as OP, resnetv2 as OR  # noqa: E402

IMG, SEED0, IMG_SEED0 = 112, 4000, 9000
RATIOS = (0.015, 0.03, 0.06, 0.12)
BUDGET, DROPOUT, EPS = 0.12, 1, 4.0


def image(i):
    return torch.rand(1, 3, IMG, IMG, generator=torch.Generator().manual_seed(IMG_SEED0 + i))


def seed_all(s):
    random.seed(s)
    torch.manual_seed(s)
    np.random.seed(s)


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--K", type=int, default=16)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--S", type=int, default=8)
    ap.add_argument("--eps", type=float, default=EPS, help="L2 bound of the pasted perturbation (reference default 4)")
    ap.add_argument("--perturb", type=float, default=0.0,
                    help="NOISE-FLOOR run: every image += perturb * N(0,1) (1e-7: below any arithmetic difference between fp32 "
                         "implementations) -- how far the END METRIC of the reference's own arithmetic moves under a last-bit change")
    ap.add_argument("--out", default="attack_success_golden.npz")
    ap.add_argument("--save-adv", type=int, default=1, help="keep the final adversarial images (frozen-patch evaluation parity)")
    a = ap.parse_args()
    K, iters, S, eps, perturb = a.K, a.iters, a.S, a.eps, a.perturb
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    params = OR.random_init(seed=0, affine_jitter=0.1)
    net = OR.OracleNet(params, weights_require_grad=False).eval()
    rec = dict(y=[], pred_adv=[], pc_pred=[], pc_cert=[], mask_frac=[], l2=[], steps=[], adv_delta=[], margin=[])
    t0 = time.time()
    for i in range(K):
        x = image(i)
        if perturb:
            x = (x + perturb * torch.randn(x.shape, generator=torch.Generator().manual_seed(77 + i))).clamp(0, 1)
        with torch.no_grad():
            y = int(net(x).argmax(-1))
        seed_all(SEED0 + i)
        trace = []
        m, p = OA.generate(net, x, BUDGET, 1000, save_dir=None, batch_id=i, targeted=False, max_iterations=iters,
                           dropout=DROPOUT, sampling_size=S, eps=eps, trace=trace)
        delta = OA.clip_paste(m, p, x, eps)
        adv = x + delta
        with torch.no_grad():
            lg = net(adv)[0]
        pa = int(lg.argmax(-1))
        top2 = torch.topk(lg, 2).values
        preds, certs = [], []
        for r in RATIOS:
            pr, ce, _, _ = OP.robust_predict(net, adv[0], IMG, r, certify=True)
            preds.append(int(pr)); certs.append(bool(ce))
        rec["y"].append(y); rec["pred_adv"].append(pa); rec["pc_pred"].append(preds); rec["pc_cert"].append(certs)
        rec["mask_frac"].append(float(m.mean())); rec["l2"].append(float(delta.norm())); rec["steps"].append(len(trace))
        rec["margin"].append(float(top2[0] - top2[1]))
        if a.save_adv:
            d = adv[0].numpy() - image(i)[0].numpy()
            assert np.array_equal(image(i)[0].numpy() + d, adv[0].numpy())
            rec["adv_delta"].append(d)
        print("img %2d  y %3d  adv %3d (top-2 margin %.2e)  PC %s cert %s  mask %.4f  l2 %.3f  steps %d  (%.0f s)" % (
            i, y, pa, rec["margin"][-1], preds, [int(c) for c in certs], rec["mask_frac"][-1], rec["l2"][-1], len(trace), time.time() - t0),
            flush=True)
    out = {k: np.asarray(v) for k, v in rec.items() if len(v)}
    out.update(K=K, iters=iters, S=S, img=IMG, seed0=SEED0, img_seed0=IMG_SEED0, ratios=np.asarray(RATIOS),
               budget=BUDGET, dropout=DROPOUT, eps=eps, perturb=perturb)
    np.savez_compressed(os.path.join(HERE, a.out), **out)
    y = out["y"]
    print("robust acc %.1f%%  acc@PC %s  cert_acc %s  cert_asr %s" % (
        (out["pred_adv"] == y).mean() * 100, (out["pc_pred"] == y[:, None]).mean(0) * 100,
        ((out["pc_pred"] == y[:, None]) & out["pc_cert"]).mean(0) * 100,
        ((out["pc_pred"] != y[:, None]) & out["pc_cert"]).mean(0) * 100))


if __name__ == "__main__":
    main()
