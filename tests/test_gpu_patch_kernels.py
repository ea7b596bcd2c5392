"""Operator-level parity of the patch side of the hot loop, which the whole-step tests only see through loose tolerances:

  K1   expand_kernel, the fused variant dp_attack_grad launches (dp_expand_step_dev) and the plain one the scan and
       PatchCleanser launch (dp_expand_dev), bit for bit against separate torch ops, at every launch shape: tile rows,
       sample groups (empty ones included), both store paths, the uncached-rectangle branch, launches that split images;
  K1^T reduce_kernel (dp_debug_k1t) against fp64, across the rectangle-batch loop and launch sequences whose first
       launch of an image overwrites G and later ones add (the bf16 fused stem-dgrad reduce, through the same hook and
       launch sequences: tests/test_gpu_ops.py);
  K4   cw_kernel (dp_debug_cw) against the reference's CW_loss (attack.py:16-23) with autograd, at ties, the -1e4 label
       slot, +-inf and NaN.

The restatements every GPU test relies on are pinned first, on CPU (the tests without the gpu mark)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import attack as OA, masks as OM

gpu = pytest.mark.gpu
DEV = "cuda:0"
NAN = float("nan")


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _rand(shape, seed):
    return torch.rand(shape, generator=torch.Generator().manual_seed(seed))


# =====================================================================================================================
# restatements (device-agnostic torch; one op per rounding, so nothing can contract into an FMA)
# =====================================================================================================================
def keep_from_rects(rects, H, W, device="cpu"):
    """int16 [n,4,4] rectangles (r0, r1, c0, c1: rows [r0,r1) x cols [c0,c1) occluded, empty when r1 <= r0 or c1 <= c0)
    -> bool keep masks [n,1,H,W] (True = keep), as attack.py:206 builds them from the mask universe."""
    r = torch.as_tensor(np.asarray(rects, np.int64).reshape(-1, 4, 4), device=device)
    rows, cols = torch.arange(H, device=device), torch.arange(W, device=device)
    in_r = (rows >= r[:, :, 0:1]) & (rows < r[:, :, 1:2])                     # [n,4,H]
    in_c = (cols >= r[:, :, 2:3]) & (cols < r[:, :, 3:4])                     # [n,4,W]
    return ~(in_r[:, :, :, None] & in_c[:, :, None, :]).any(1)[:, None]


def paste_ref(x, mask, pattern, scale):
    """attack.py:184-185 / utils.py:105-110 with the clip scale given: x + (mask * (pattern - x)) * scale[b]."""
    d = pattern - x
    d = mask * d
    d = d * scale.view(-1, 1, 1, 1)
    return x + d


def k1_ref(adv_b, keep, cp, dtype):
    """One image [3,H,W] in [0,1] and its samples' keep masks [s,1,H,W] -> network input [s,H,W,cp] in `dtype`:
    occlude to 0.5 (attack.py:206), (v - 0.5) / 0.5 (utils.py:77-78), NHWC, round to dtype, pad channels exactly 0."""
    v = OA.occlude(adv_b[None], keep)
    v = (v - 0.5) * 2.0
    v = v.permute(0, 2, 3, 1).to(dtype)
    out = torch.zeros(v.shape[:3] + (cp,), dtype=dtype, device=v.device)
    out[..., :3] = v
    return out


def k1t_ref(dz, keep, B, S):
    """K1^T in fp64: G[b] = 2 * sum_s keep_s * dz_s[..., :3] (NHWC -> NCHW) over all B*S samples, with per element the
    number m of samples summed into it and sum_s keep_s * |2 dz_s| (the two terms of the recursive-summation bound)."""
    H, W = dz.shape[1], dz.shape[2]
    d = dz[..., :3].double().permute(0, 3, 1, 2) * 2.0 * keep.double()
    m = keep.double().reshape(B, S, 1, H, W).sum(1)
    return d.reshape(B, S, 3, H, W).sum(1), m, d.abs().reshape(B, S, 3, H, W).sum(1)


def cw_ref(logits, y, targeted, confidence, w):
    """attack.py:16-23 (oracle.attack.cw_loss), rows grouped by criterion; autograd gives w * d loss / d logits; preds
    are torch.argmax.  -> (loss [N], preds [N], dlogits [N,K]) on CPU, fp32."""
    lg = logits.detach().cpu().clone().requires_grad_(True)
    N, K = lg.shape
    y = torch.as_tensor(y, dtype=torch.int64)
    tg = torch.as_tensor(np.asarray(targeted, bool))
    loss = torch.empty(N)
    total = 0.0
    for crit in (False, True):
        sel = torch.nonzero(tg == crit).view(-1)
        if len(sel):
            lv = OA.cw_loss(lg[sel], y[sel], K, crit, confidence)
            loss[sel] = lv.detach()
            total = total + (lv * w).sum()
    total.backward()
    return loss, lg.detach().argmax(1), lg.grad


def cw_bound(logits, y, confidence):
    """The kernel adds conf + (other - real), the reference (conf + other) - real: a few fp32 roundings of
    |conf| + |other| + |real| apart."""
    lg = logits.detach().cpu()
    oh = F.one_hot(torch.as_tensor(y, dtype=torch.int64), lg.shape[1]).float()
    real = (lg * oh).sum(1)
    other = ((1.0 - oh) * lg - oh * 1e4).max(1)[0]
    return 2.0 ** -22 * (abs(confidence) + other.abs() + real.abs())


def k1_expected_shape(H, W, cp, es, fused, n0, n, S, num_sms, rows=0, sg=0):
    """The launch rule of kernels_patch.cu (expand_launch): (tile rows R, sample groups) for a launch of samples
    [n0, n0+n).  A forced R that does not divide H or needs more than 200 KB of shared memory falls back to the rule."""
    np_ = 7 if fused else 3
    nb_img = (n0 + n - 1) // S - n0 // S + 1

    def usable(r):
        return 1 <= r <= 32 and H % r == 0 and 512 + 2048 + np_ * r * W * 4 + r * W * cp * es <= 200 * 1024
    if rows > 0 and usable(rows):
        R = rows
    else:
        R = 0
        for r in (8, 7, 4, 2, 1):
            if usable(r):
                R = R or r
                if nb_img * (H // r) >= 4 * num_sms or r <= 4:
                    R = r
                    break
        R = R or 1
    if sg > 0:
        return R, sg
    g = 1
    while nb_img * (H // R) * g < 2 * num_sms and g * 2 * 8 <= S and g < 32:
        g *= 2
    return R, g


def special_rects(H):
    """Rectangles where the expand kernel's tile / row / 16-byte-chunk logic can go wrong; int16 [n,4,4]."""
    W = H
    cases = [
        [],                                                            # no occluder
        [(0, H, 0, W)],                                                # the whole image
        [(0, 5, 3, 20)], [(H - 6, H, 10, 30)],                         # touching row 0 / row H
        [(9, 30, 0, 4)], [(20, 41, W - 5, W)],                         # touching column 0 / column W
        [(H - 1, H, W - 3, W)], [(5, 6, 0, W)],                        # last row's last pixels; one full row
    ]
    cases += [[(3, H - 3, c0, c0 + 1)] for c0 in range(8)]            # 1 px wide: every edge position in a 16-byte chunk
    cases += [
        [(8, 16, 5, 9), (14, 28, 30, 40), (7, 21, 44, 50), (16, 32, 12, 13)],   # on the tile-row boundaries of R = 8, 14, 7, 16
        [(4, 30, 4, 30), (10, 40, 10, 40), (20, 50, 2, 22), (1, 12, 25, 52)],   # four overlapping
        [(30, 10, 5, 20)], [(10, 30, 20, 5)],                                    # degenerate: r1 <= r0 / c1 <= c0
        [(12, 12, 0, W), (0, H, 7, 7)],                                          # zero height / zero width
    ]
    out = np.zeros((len(cases), 4, 4), np.int16)
    for i, rs in enumerate(cases):
        for k, r in enumerate(rs):
            out[i, k] = r
    return out


def mixed_rects(H, B, S, seed):
    """[B*S,4,4]: every special rectangle set once, the rest double masks of the universe (dual for every other sample,
    gathered as bench.py does), shuffled over the images."""
    from dorpatch_b200 import masks as PM
    sp = special_rects(H)
    table = PM.universe(H, 2)
    rng = np.random.RandomState(seed)
    N = B * S
    n_uni = max(0, N - len(sp))
    uni = PM.gather(table, rng.randint(0, len(table), n_uni), rng.randint(0, len(table), n_uni))
    uni[1::2, 2:] = 0
    allr = np.concatenate([sp, uni])[:N]
    return np.ascontiguousarray(allr[rng.permutation(N)])


# =====================================================================================================================
# CPU self-checks of the restatements
# =====================================================================================================================
def test_keep_from_rects_matches_oracle_masks():
    """The rectangle decoder equals the oracle's materialised universe (PatchCleanser.py:44-59) and numpy slicing on the
    special rectangles (degenerate ones are empty, as r0:r1 with r1 <= r0 is)."""
    H = 56
    pairs = OM.universe_rects(H, 2)
    got = keep_from_rects(np.pad(OM.rects_to_array(pairs), ((0, 0), (0, 2), (0, 0))), H, H)
    assert torch.equal(got, torch.from_numpy(OM.rects_to_bool(pairs, H)))
    sp = special_rects(H)
    ref = np.ones((len(sp), 1, H, H), bool)
    for i, rs in enumerate(sp):
        for r0, r1, c0, c1 in rs:
            ref[i, 0, r0:r1, c0:c1] = False
    assert torch.equal(keep_from_rects(sp, H, H), torch.from_numpy(ref))
    assert ref[0].all() and not ref[1].any()


@pytest.mark.parametrize("cp,dtype", [(4, torch.float32), (3, torch.bfloat16)])
def test_k1_reference_equals_oracle_clip_occlude_normalise(cp, dtype):
    """paste_ref + k1_ref == x + oracle.clip_paste, oracle.occlude, (v - 0.5) / 0.5, NHWC, bit for bit, when given the
    oracle's own clip scale -- including scale < 1, scale == 1 (||delta|| < eps) and zero delta (eps / 0 -> 1)."""
    H, B, S, eps = 56, 3, 8, 4.0
    x, m, p = _rand((B, 3, H, H), 1), _rand((B, 1, H, H), 2), _rand((B, 3, H, H), 3)
    m[1] *= 0.01
    m[2] = 0.0
    scale = (eps / torch.norm(m * (p - x), p=2, dim=(1, 2, 3))).clamp(max=1.0)
    assert scale[0] < 1 and scale[1] == 1 and scale[2] == 1
    rects = mixed_rects(H, B, S, 0)
    keep = keep_from_rects(rects, H, H).reshape(B, S, 1, H, H)
    adv_o = x + OA.clip_paste(m, p, x, eps)
    norm_o = ((OA.occlude(adv_o[:, None], keep) - 0.5) / 0.5).reshape(B * S, 3, H, H).permute(0, 2, 3, 1)
    adv = paste_ref(x, m, p, scale)
    assert torch.equal(adv, adv_o)
    got = torch.cat([k1_ref(adv[b], keep[b], cp, dtype) for b in range(B)])
    assert torch.equal(got[..., :3], norm_o.to(dtype)) and (got[..., 3:] == 0).all()


def test_k1t_reference_equals_loops():
    """k1t_ref against the plain loop G[b,c,h,w] = sum over the image's samples that keep (h,w) of 2 dz[s,h,w,c]."""
    H, B, S, cpd = 8, 2, 3, 4
    dz = torch.randn(B * S, H, H, cpd, generator=torch.Generator().manual_seed(4))
    dz[..., 3] = NAN
    rects = np.zeros((B * S, 4, 4), np.int16)
    rects[0, 0] = (1, 5, 2, 7)
    rects[1, :2] = [(0, 8, 0, 8), (3, 4, 3, 4)]
    rects[4, 0], rects[4, 1] = (2, 3, 0, 8), (0, 8, 6, 7)
    keep = keep_from_rects(rects, H, H)
    ref, m, absum = k1t_ref(dz, keep, B, S)
    G, M, A = np.zeros((B, 3, H, H)), np.zeros((B, 1, H, H)), np.zeros((B, 3, H, H))
    for n in range(B * S):
        b = n // S
        for h in range(H):
            for w in range(H):
                if not bool(keep[n, 0, h, w]):
                    continue
                M[b, 0, h, w] += 1
                for c in range(3):
                    G[b, c, h, w] += 2.0 * float(dz[n, h, w, c])
                    A[b, c, h, w] += abs(2.0 * float(dz[n, h, w, c]))
    assert np.allclose(ref.numpy(), G, rtol=1e-12, atol=0) and np.array_equal(m.numpy(), M) and np.allclose(absum.numpy(), A, rtol=1e-12)


def test_cw_reference_equals_loop():
    """cw_ref (oracle CW_loss + autograd) against a plain per-row loop on finite logits with ties: real = l[y], other =
    the first maximum of the logits with the label slot set to -1e4, loss = clamp(margin, 0) in the reference's
    association, gradient +-w to the label and to other's index (none when other is the label slot) where the clamp's
    input is >= 0."""
    K, w = 7, np.float32(1 / 3)
    rng = np.random.RandomState(5)
    rows = [rng.randn(K).astype(np.float32) for _ in range(6)]
    rows[1][[2, 4]] = 9.0                                    # tie for the max
    rows[2][:] = -2e4; rows[2][3] = 1.0                      # every non-label logit below -1e4
    rows[3][:] = -3e4; rows[3][1] = -1e4                     # tie with the label slot at -1e4, lower index than y
    rows[4][:] = -3e4; rows[4][6] = -1e4                     # ... higher index than y
    rows[5][:] = 0.0; rows[5][3] = -0.5                      # untargeted, conf 0.5: pre exactly 0
    logits = torch.from_numpy(np.stack(rows))
    y = [3, 0, 3, 3, 3, 3]
    tg = [False, True, False, True, False, False]
    for conf in (0.0, 0.5):
        loss, preds, dl = cw_ref(logits, y, tg, conf, float(w))
        for i, l in enumerate(rows):
            cand = np.where(np.arange(K) == y[i], np.float32(-1e4), l)
            oi = int(np.argmax(cand))
            other, real = cand[oi], l[y[i]]
            pre = (np.float32(conf) + other) - real if tg[i] else (np.float32(conf) + real) - other
            assert loss[i].item() == max(pre, np.float32(0)), (i, conf)
            g = np.zeros(K, np.float32)
            if pre >= 0:
                g[y[i]] = -w if tg[i] else w
                if oi != y[i]:
                    g[oi] += w if tg[i] else -w
            assert np.array_equal(dl[i].numpy(), g), (i, conf, dl[i], g)
            assert preds[i].item() == int(np.argmax(l))
        if conf == 0.5:                                      # pre == 0: zero loss, and the clamp passes the gradient
            assert loss[5] == 0 and dl[5].abs().sum() > 0


def test_k1_launch_rule_restatement_table():
    """k1_expected_shape at 148 SMs gives the shapes the rule was tuned to (profiles/r02_k1_sweep.txt): 4-row tiles and
    8 sample groups for B=1 x S=128, 8-row tiles for the whole c3 step, 4 x 1 (128 samples per item: the uncached
    rectangle branch) for B=8 x S=128, 4 x 1 for the B=2 x S=3 step at 112 px."""
    for fused in (True, False):
        for cp, es in ((4, 4), (3, 2)):
            assert k1_expected_shape(224, 224, cp, es, fused, 0, 128, 128, 148) == (4, 8)
            assert k1_expected_shape(224, 224, cp, es, fused, 0, 2048, 32, 148) == (8, 1)
            assert k1_expected_shape(224, 224, cp, es, fused, 0, 1024, 128, 148) == (4, 1)
            assert k1_expected_shape(112, 112, cp, es, fused, 0, 6, 3, 148) == (4, 1)
    assert k1_expected_shape(56, 56, 4, 4, True, 0, 36, 12, 148, rows=16, sg=3) == (4, 3)      # 16 does not divide 56


# =====================================================================================================================
# GPU: K1
# =====================================================================================================================
@pytest.fixture
def k1_tuning():
    """dp_debug_k1_tuning is process-wide: always hand the launch shape back to the rule."""
    from dorpatch_b200 import _lib
    lib = _lib.load()
    yield lib
    lib.dp_debug_k1_tuning(0, 0, 0)


def _k1_last(lib):
    v = (C.c_int32 * 4)()
    assert lib.dp_debug_k1_last(C.cast(v, C.c_void_p)) == 0
    return tuple(v)


def _num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _engine_dtype(e):
    return torch.bfloat16 if e.elem_bytes == 2 else torch.float32


def _bits(t):
    return t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


def _step_inputs(B, H, seed):
    """x, mask, pattern on the device; image b % 3 == 1 has ||delta|| < eps (scale 1), b % 3 == 2 a zero delta."""
    x, m, p = _rand((B, 3, H, H), seed), _rand((B, 1, H, H), seed + 1), _rand((B, 3, H, H), seed + 2)
    m[1::3] *= 0.01
    m[2::3] = 0.0
    return x.to(DEV), m.to(DEV), p.to(DEV)


def _paste_scale(e, x, m, p, eps=4.0):
    """The step's paste (dp_paste with no output buffer): writes the clip scale the fused K1 reads, and returns it."""
    B = x.shape[0]
    sc = np.empty(B, np.float32)
    from dorpatch_b200 import _lib
    _lib.check(e.lib.dp_paste(e.handle, _ptr(x), _ptr(m), _ptr(p), B, eps, None, None, C.c_void_p(sc.ctypes.data), e._stream()))
    return torch.from_numpy(sc).to(DEV)


def _launch_fused(e, x, m, p, B, S, rects_d, n0, n, out):
    from dorpatch_b200 import _lib
    _lib.check(e.lib.dp_expand_step_dev(e.handle, _ptr(x), _ptr(m), _ptr(p), B, S, _ptr(rects_d), n0, n, _ptr(out), e._stream()))


def _launch_plain(e, img, B, S, rects_d, out):
    from dorpatch_b200 import _lib
    _lib.check(e.lib.dp_expand_dev(e.handle, _ptr(img), B, S, _ptr(rects_d), _ptr(out), e._stream()))


def _nan_out(e, n):
    return torch.full((n, e.img, e.img, e.c_pad), NAN, dtype=_engine_dtype(e), device=DEV)


def _check_against_ref(out, adv, keep, B, S, cp, dtype, n0=0):
    """out holds samples [n0, n0 + len(out)); compare image by image (the reference stays one image large)."""
    n1 = n0 + out.shape[0]
    for b in range(n0 // S, (n1 - 1) // S + 1):
        lo, hi = max(n0, b * S), min(n1, (b + 1) * S)
        ref = k1_ref(adv[b], keep[lo:hi], cp, dtype)
        got = out[lo - n0:hi - n0]
        if not torch.equal(_bits(got), _bits(ref)):
            bad = (_bits(got) != _bits(ref)).nonzero()
            raise AssertionError("image %d: %d elements differ, first [sample, h, w, c] = %s (got %s, want %s)" % (
                b, bad.shape[0], (bad[0] + torch.tensor([lo, 0, 0, 0], device=bad.device)).tolist(),
                got[tuple(bad[0])].item(), ref[tuple(bad[0])].item()))


K1_ROWS = (1, 2, 4, 7, 8, 14, 16)
K1_SG = (1, 2, 3, 8, 13)                    # S = 12 samples per image: 13 groups leave one empty


@gpu
@pytest.mark.parametrize("fused", [True, False], ids=["fused", "plain"])
@pytest.mark.parametrize("H", [56, 224])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_k1_bit_exact_at_every_launch_shape(engine_factory, k1_tuning, precision, H, fused):
    """K1 at every forced launch shape (tile rows x sample groups x store path) equals the separate-op restatement bit
    for bit, on every special rectangle, with every output pre-filled with NaN (a sample the kernel never writes
    fails).  dp_debug_k1_last must report the requested shape, or the rule's when the request is unusable."""
    e = engine_factory(img=H, precision=precision, chunk=8, max_images=64)
    B, S = 3, 12
    N = B * S
    dt, cp = _engine_dtype(e), e.c_pad
    x, m, p = _step_inputs(B, H, 10)
    rects = mixed_rects(H, B, S, 1)
    rects_d = torch.from_numpy(rects).to(DEV)
    keep = keep_from_rects(rects, H, H, DEV)
    if fused:
        scale = _paste_scale(e, x, m, p)
        assert scale[0] < 1 and scale[1] == 1 and scale[2] == 1
        adv = paste_ref(x, m, p, scale)
    else:
        adv = x
    refs = torch.cat([k1_ref(adv[b], keep[b * S:(b + 1) * S], cp, dt) for b in range(B)])
    nsm = _num_sms()
    seen = set()
    for mode in (0, 1):
        for rows in K1_ROWS:
            for sg in K1_SG:
                k1_tuning.dp_debug_k1_tuning(rows, sg, mode)
                out = _nan_out(e, N)
                if fused:
                    _launch_fused(e, x, m, p, B, S, rects_d, 0, N, out)
                else:
                    _launch_plain(e, x, B, S, rects_d, out)
                last = _k1_last(k1_tuning)
                want = k1_expected_shape(H, H, cp, e.elem_bytes, fused, 0, N, S, nsm, rows, sg)
                assert last[:2] == want, (rows, sg, mode, last, want)
                seen.add((last[0], last[1], mode))
                if not torch.equal(_bits(out), _bits(refs)):
                    _check_against_ref(out, adv, keep, B, S, cp, dt)
                    raise AssertionError("mismatch at rows %d sg %d mode %d" % (rows, sg, mode))
    print("K1 %s %s H=%d: launch shapes (R, sg, mode) run: %s" % ("fused" if fused else "plain", precision, H, sorted(seen)))


# (B, S, H, forced rows, forced mode): the automatic rule at production shapes, and the shape DESIGN.md section 4 set aside
K1_PRODUCTION = {
    "B1xS128": (1, 128, 224, 0, 0),
    "B64xS32": (64, 32, 224, 0, 0),
    "B8xS128": (8, 128, 224, 0, 0),
    "B2xS3_112px": (2, 3, 112, 0, 0),
    "B64xS32_R14_mode1": (64, 32, 224, 14, 1),
}


@gpu
@pytest.mark.parametrize("case", list(K1_PRODUCTION))
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_k1_fused_bit_exact_at_production_shapes(engine_factory, k1_tuning, precision, case):
    """The fused K1 as dp_attack_grad launches it for a whole step, at the shapes the automatic rule picks in
    production: 8 sample groups for B=1 x S=128, 8-row tiles for the c3 step, the uncached-rectangle branch (128 samples
    per work item) for B=8 x S=128, the small-step shape -- and forced 14-row tiles with 16-byte stores only."""
    B, S, H, rows, mode = K1_PRODUCTION[case]
    if rows and precision != "fp32":
        pytest.skip("the set-aside shape is checked on the fp32 engine")
    e = engine_factory(img=H, precision=precision, chunk=8, max_images=64)
    N = B * S
    dt, cp = _engine_dtype(e), e.c_pad
    x, m, p = _step_inputs(B, H, 20)
    rects = mixed_rects(H, B, S, 2)
    rects_d = torch.from_numpy(rects).to(DEV)
    scale = _paste_scale(e, x, m, p)
    adv = paste_ref(x, m, p, scale)
    k1_tuning.dp_debug_k1_tuning(rows, 0, mode)
    out = _nan_out(e, N)
    _launch_fused(e, x, m, p, B, S, rects_d, 0, N, out)
    last = _k1_last(k1_tuning)
    want = k1_expected_shape(H, H, cp, e.elem_bytes, True, 0, N, S, _num_sms(), rows, 0)
    print("K1 fused %s %s: launch shape (R, sg, grid, CTAs/SM) = %s, rule %s, %d SMs" % (precision, case, last, want, _num_sms()))
    assert last[:2] == want, (last, want)
    keep = keep_from_rects(rects, H, H, DEV)
    _check_against_ref(out, adv, keep, B, S, cp, dt)


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("B,S,H,step", [(3, 5, 56, 4), (2, 128, 56, 100), (2, 128, 224, 100)])
def test_k1_fused_chunk_offset_launches(engine_factory, k1_tuning, precision, B, S, H, step):
    """Launches [n0, n0 + step) that split images, each into its own buffer, concatenate to the single whole-step launch
    bit for bit and both equal the restatement -- under the rule's shape and under forced sample groups / store path."""
    e = engine_factory(img=H, precision=precision, chunk=8, max_images=64)
    N = B * S
    dt, cp = _engine_dtype(e), e.c_pad
    x, m, p = _step_inputs(B, H, 30)
    rects = mixed_rects(H, B, S, 3)
    rects_d = torch.from_numpy(rects).to(DEV)
    adv = paste_ref(x, m, p, _paste_scale(e, x, m, p))
    keep = keep_from_rects(rects, H, H, DEV)
    for rows, sg, mode in ((0, 0, 0), (4, 3, 0), (4, 1, 0), (8, 2, 1)):     # sg 1: up to `step` samples per item, uncached
        k1_tuning.dp_debug_k1_tuning(rows, sg, mode)
        whole = _nan_out(e, N)
        _launch_fused(e, x, m, p, B, S, rects_d, 0, N, whole)
        shapes = [_k1_last(k1_tuning)]
        parts = []
        for n0 in range(0, N, step):
            n = min(step, N - n0)
            part = _nan_out(e, n)
            _launch_fused(e, x, m, p, B, S, rects_d, n0, n, part)
            shapes.append(_k1_last(k1_tuning))
            want = k1_expected_shape(H, H, cp, e.elem_bytes, True, n0, n, S, _num_sms(), rows, sg)
            assert shapes[-1][:2] == want, (n0, n, shapes[-1], want)
            _check_against_ref(part, adv, keep, B, S, cp, dt, n0)
            parts.append(part)
        print("K1 fused %s B=%d S=%d H=%d launches of %d, forced (%d, %d, mode %d): shapes %s" % (
            precision, B, S, H, step, rows, sg, mode, [s[:2] for s in shapes]))
        assert torch.equal(_bits(torch.cat(parts)), _bits(whole))
        _check_against_ref(whole, adv, keep, B, S, cp, dt)


# =====================================================================================================================
# GPU: K1^T
# =====================================================================================================================
@pytest.fixture(scope="module")
def cudnn_stem_bwd_engine(oracle_params):
    """bf16 engine whose K1^T is reduce_kernel on cuDNN's stem dgrad (DORPATCH_STEM_BWD=cudnn: bf16 dz, 8 channels)."""
    from dorpatch_b200.engine import Engine
    os.environ["DORPATCH_STEM_BWD"] = "cudnn"
    try:
        e = Engine(img=56, precision="bf16", chunk=8, max_images=4, autotune=False)
    finally:
        os.environ.pop("DORPATCH_STEM_BWD", None)
    e.load_state_dict(oracle_params)
    yield e
    e.close()


def _k1t_rects(H, B, S, seed):
    """Universe double masks; every 7th sample fully occluded, every 11th without an occluder."""
    from dorpatch_b200 import masks as PM
    table = PM.universe(H, 2)
    rects = PM.gather(table, np.random.RandomState(seed).randint(0, len(table), B * S))
    rects[::7] = 0
    rects[::7, 0] = (0, H, 0, H)
    rects[5::11] = 0
    return np.ascontiguousarray(rects)


def _run_k1t(e, dz, rects, B, S, step, G):
    """K1^T over [0, B*S) in launches of `step` samples, each launch reading its slice of dz."""
    N = B * S
    rp = C.c_void_p(rects.ctypes.data) if rects is not None else None
    from dorpatch_b200 import _lib
    for n0 in range(0, N, step):
        n = min(step, N - n0)
        _lib.check(e.lib.dp_debug_k1t(e.handle, _ptr(dz[n0:n0 + n]), rp, B, S, n0, n, _ptr(G), e._stream()))
    torch.cuda.synchronize()


K1T_CASES = {   # (B, S, samples per launch, rectangles?)
    "S1": (3, 1, 3, True),
    "S3": (2, 3, 6, True),
    "S128": (2, 128, 256, True),
    "S129": (2, 129, 258, True),
    "S300": (2, 300, 600, True),
    "S300_launches_of_128": (2, 300, 128, True),
    "S5_launches_of_4": (3, 5, 4, True),
    "S129_launches_of_50": (2, 129, 50, True),
    "S130_no_rects": (2, 130, 260, False),
}


@gpu
@pytest.mark.parametrize("case", list(K1T_CASES))
@pytest.mark.parametrize("engine_kind", ["fp32", "bf16_cudnn_stem_bwd"])
def test_k1t_reduce_vs_fp64(engine_factory, cudnn_stem_bwd_engine, engine_kind, case):
    """reduce_kernel (K1^T of the fp32 / tf32 engines, and of bf16 with DORPATCH_STEM_BWD=cudnn) against fp64, element by
    element within the recursive-summation bound |got - ref| <= 2 m 2^-24 sum|2 dz| (m = samples summed into the element):
    a dropped or doubled sample breaks it by orders of magnitude.  Around the 128-sample rectangle batch, across launch
    sequences that split images (G starts as NaN: an image's first launch must overwrite it, later ones add), with fully
    occluded samples (exactly 0), without rectangles, and with NaN / 1e30 in the pad channels (never read)."""
    B, S, step, with_rects = K1T_CASES[case]
    if engine_kind == "fp32":
        e, dt, cpd = engine_factory(img=56, precision="fp32", chunk=8, max_images=64), torch.float32, 4
    else:
        e, dt, cpd = cudnn_stem_bwd_engine, torch.bfloat16, 8
    H, N = e.img, B * S
    dz = torch.rand(N, H, H, cpd, generator=torch.Generator().manual_seed(40)) * 2 - 1
    dz[0::2, :, :, 3:] = NAN
    dz[1::2, :, :, 3:] = 1e30
    dz = dz.to(dt).to(DEV)
    rects = _k1t_rects(H, B, S, 41) if with_rects else None
    if case == "S3":
        rects[S:] = 0
        rects[S:, 0] = (0, H, 0, H)                        # image 1: every sample fully occluded
    keep = keep_from_rects(rects, H, H, DEV) if with_rects else torch.ones(N, 1, H, H, dtype=torch.bool, device=DEV)
    ref, mcount, absum = k1t_ref(dz, keep, B, S)
    G = torch.full((B, 3, H, H), NAN, device=DEV)
    _run_k1t(e, dz, rects, B, S, step, G)
    err = (G.double() - ref).abs()
    bound = 2.0 * mcount * 2.0 ** -24 * absum + 1e-30
    worst = float((err / bound).max())
    print("K1^T %s %s: max |err| / bound = %.3f, max |err| = %.2e" % (engine_kind, case, worst, float(err.max())))
    assert torch.isfinite(G).all()
    assert (err <= bound).all(), worst
    if case == "S3":
        assert (G[1] == 0).all()


# =====================================================================================================================
# GPU: K4
# =====================================================================================================================
def cw_cases(K, confidence, seed):
    """(logits [N,K] fp32, y [N], targeted [N]): rows at the kernel's edges, N not a multiple of 8."""
    rng = np.random.RandomState(seed)
    conf = np.float32(confidence)
    rows, ys, tgs = [], [], []

    def add(row, y, tg):
        rows.append(np.asarray(row, np.float32)); ys.append(y); tgs.append(tg)
    lo = K // 3
    for tg in (False, True):
        r = rng.randn(K); y = K - 1; r[y] = r.max() + 1.0; add(r, y, tg)           # label the unique max
        r = rng.randn(K); y = 0; r[y] = r.min() - 1.0; add(r, y, tg)               # label not the max
        r = rng.randn(K); r[[1, K - 2]] = 7.5; add(r, K // 2, tg)                  # tie for the max (and for other)
        r = rng.randn(K); r[[lo, K - 1]] = 7.5; add(r, K - 1, tg)                  # the label ties the max at a higher index
        r = -2e4 - rng.rand(K) * 1e4; y = lo; r[y] = 3.0; add(r, y, tg)            # every non-label logit below -1e4
        r = np.full(K, -3e4); r[0] = -1e4; add(r, lo, tg)                          # -1e4 exactly, below the label's index
        r = np.full(K, -3e4); r[K - 1] = -1e4; add(r, lo, tg)                      # -1e4 exactly, above the label's index
        r = rng.randn(K) - 5.0; y = lo                                              # pre exactly 0: the gradient passes
        if tg:
            r[y], r[0] = conf, 0.0
        else:
            r[y], r[0] = 0.0, conf
        add(r, y, tg)
        r = rng.randn(K); r[K - 1] = np.inf; add(r, 0, tg)                         # +inf elsewhere
        r = rng.randn(K); r[lo] = -np.inf; add(r, 0, tg)                           # -inf elsewhere
        r = rng.randn(K); r[lo] = np.inf; add(r, lo, tg)                           # +inf at the label
        r = np.full(K, -np.inf); add(r, lo, tg)                                    # all -inf: argmax 0
        r = rng.randn(K); r[0] = 50.0; r[K - 1] = np.nan; add(r, 0, tg)           # one NaN: argmax is its index
        r = rng.randn(K); r[[lo, K - 1]] = np.nan; add(r, K - 1, tg)              # two NaNs: the first
        add(np.full(K, np.nan), lo, tg)                                            # all NaN
    add(rng.randn(K), 1, False)                                                    # N = 31
    return torch.from_numpy(np.stack(rows)), np.array(ys, np.int32), np.array(tgs, np.uint8)


def _cw_launch(e, logits, y, tg, confidence, w, with_loss=True):
    from dorpatch_b200 import _lib
    N, K = logits.shape
    ld = logits.to(DEV).contiguous()
    preds = torch.full((N,), -7, dtype=torch.int32, device=DEV)
    loss = torch.full((N,), -7.0, device=DEV) if with_loss else None
    dl = torch.full((N, K), NAN, device=DEV) if with_loss else None
    yd = torch.from_numpy(y).to(DEV) if with_loss else None
    td = torch.from_numpy(tg).to(DEV) if with_loss else None
    _lib.check(e.lib.dp_debug_cw(e.handle, _ptr(ld), _ptr(yd), _ptr(td), float(confidence), float(w), _ptr(loss), _ptr(preds),
                                 _ptr(dl), N, K, e._stream()))
    torch.cuda.synchronize()
    return (loss.cpu() if with_loss else None), preds.cpu().long(), (dl.cpu() if with_loss else None)


@gpu
@pytest.mark.parametrize("K", [10, 33, 1000])
@pytest.mark.parametrize("confidence", [0.0, 0.1])
def test_cw_kernel_vs_reference_cw_loss(engine_factory, K, confidence):
    """K4 against attack.py:16-23 restated in torch (oracle.attack.cw_loss) with autograd: preds (torch.argmax: lowest
    index on ties, the first NaN) and the dlogits positions and values exactly; the loss within a few fp32 roundings of
    |conf| + |other| + |real| (the kernel adds in a different order) -- NaN exactly where the reference's one-hot product
    gives NaN (any non-finite logit in the row), with a zero gradient there.  Also N = 1 and the argmax-only launch
    that dp_predict runs."""
    e = engine_factory(img=56, precision="fp32", chunk=8, max_images=64)
    conf = float(np.float32(confidence))
    w = float(np.float32(1.0 / 3.0))
    logits, y, tg = cw_cases(K, conf, 60 + K)
    N = logits.shape[0]
    assert N % 8 != 0
    loss, preds, dl = _cw_launch(e, logits, y, tg, conf, w)
    rl, rp, rd = cw_ref(logits, y, tg, conf, w)
    bad = [i for i in range(N) if preds[i] != rp[i]]
    assert not bad, [(i, int(preds[i]), int(rp[i])) for i in bad]
    nan_ref = torch.isnan(rl)
    assert torch.equal(torch.isnan(loss), nan_ref), (torch.isnan(loss) != nan_ref).nonzero().view(-1).tolist()
    assert (loss[~nan_ref] >= 0).all()
    tol = cw_bound(logits, y, conf)
    err = (loss - rl).abs()
    assert (err[~nan_ref] <= tol[~nan_ref]).all(), [(i, loss[i].item(), rl[i].item()) for i in range(N) if not nan_ref[i] and err[i] > tol[i]]
    rows_bad = [i for i in range(N) if not torch.equal(dl[i], rd[i])]
    assert not rows_bad, [(i, dl[i].nonzero().view(-1).tolist(), rd[i].nonzero().view(-1).tolist()) for i in rows_bad]
    assert (dl[nan_ref] == 0).all()
    # N = 1
    l1, p1, d1 = _cw_launch(e, logits[:1], y[:1], tg[:1], conf, w)
    assert p1[0] == rp[0] and torch.equal(d1[0], rd[0]) and abs(l1[0] - rl[0]) <= tol[0]
    # argmax only (no labels, no loss): dp_predict's launch
    _, p2, _ = _cw_launch(e, logits, y, tg, conf, w, with_loss=False)
    assert torch.equal(p2, logits.argmax(1))
