"""Op-level GPU parity of the hand-written kernels that the network-level tests only see through the whole net:
GroupNorm(32)+ReLU v2 forward / backward (fp32 and bf16, every ResNetV2-50 shape class), the bf16 engine's fused
stem-dgrad + masked EOT reduce (K1^T as the bench runs it), and the tcgen05 GroupNorm-prologue GEMM -- each against
a PyTorch fp32/fp64 CPU restatement of the same operator on the same (bf16-rounded) operands, through the C ABI's
dp_debug_* hooks.  Restated operators: timm GroupNormAct = F.group_norm(32, eps 1e-5) + ReLU and its autograd
gradient (reference call site utils.py:77-78 -> timm resnetv2); the stem's StdConv2d 7x7/2 transposed; 1x1 StdConv2d."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import masks as OM, resnetv2 as OR

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _rand(shape, seed, scale=1.0, shift=0.0):
    return torch.rand(shape, generator=torch.Generator().manual_seed(seed)) * 2 * scale - scale + shift


@pytest.fixture(scope="module")
def engines(oracle_params):
    from dorpatch_b200.engine import Engine
    made = {}

    def get(precision):
        if precision not in made:
            e = Engine(img=224, precision=precision, chunk=8, max_images=2, autotune=False)
            e.load_state_dict(oracle_params)
            made[precision] = e
        return made[precision]
    yield get
    for e in made.values():
        e.close()


# (7056, 256) is stage 1 at 336 px: too large for v2's plan in fp32 and bf16, so it runs on the two-pass kernels
GN_SHAPES = [(3136, 64), (3136, 256), (784, 128), (784, 512), (196, 1024), (196, 256), (49, 2048), (49, 512), (7056, 256)]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("P,Cc", GN_SHAPES)
@pytest.mark.parametrize("neg_gamma", [False, True])
def test_groupnorm_relu_fwd_bwd_vs_fp64(engines, precision, P, Cc, neg_gamma):
    """y = relu(group_norm(x)) and dx = d/dx <relu(group_norm(x)), dy> (+ addend) against torch fp64 autograd.
    fp32: 2e-5 of the tensor's max; bf16 (bf16 in/out, fp32 statistics): 1/128 of the max (one bf16 ulp at the top of
    the range).  Elements whose pre-activation is within 1e-3 of the ReLU kink may gate either way and are excluded.
    neg_gamma exercises the generic-gate kernel variant (gamma <= 0 on some channels)."""
    from dorpatch_b200 import _lib
    if neg_gamma and (P, Cc) not in ((784, 128), (3136, 256), (49, 2048)):
        pytest.skip("generic-gate variant: three shape classes are enough")
    e = engines(precision)
    N = 3
    dt = torch.bfloat16 if precision == "bf16" else torch.float32
    x = _rand((N, P, Cc), 1, 1.5, 0.7).to(dt)
    dy = _rand((N, P, Cc), 2, 1.0, 0.05).to(dt)
    ad = _rand((N, P, Cc), 3, 0.5).to(dt)
    gamma = 1.0 + 0.3 * _rand((Cc,), 4)
    beta = 0.3 * _rand((Cc,), 5)
    if neg_gamma:
        gamma[1], gamma[Cc - 3] = -0.5, 0.0
    xd, dyd, add = x.to(DEV), dy.to(DEV), ad.to(DEV)
    y, dx = torch.empty_like(xd), torch.empty_like(xd)
    stats = torch.empty(N, 32, 2, device=DEV)
    gd, bd = gamma.to(DEV), beta.to(DEV)
    _lib.check(e.lib.dp_debug_gn(e.handle, _ptr(xd), _ptr(dyd), _ptr(add), _ptr(gd), _ptr(bd), 0 if neg_gamma else 1, _ptr(y), _ptr(dx),
                                 _ptr(stats), N, P, Cc, e._stream()))
    torch.cuda.synchronize()
    xr = x.double().permute(0, 2, 1).reshape(N, Cc, P, 1).requires_grad_(True)       # NCHW view of the NHWC tensor
    pre = F.group_norm(xr, 32, gamma.double(), beta.double(), 1e-5)
    yr = F.relu(pre)
    (yr * dy.double().permute(0, 2, 1).reshape(N, Cc, P, 1)).sum().backward()
    dxr = xr.grad + ad.double().permute(0, 2, 1).reshape(N, Cc, P, 1)
    sure = pre.detach().abs() > 1e-3
    got_y = y.cpu().double().permute(0, 2, 1).reshape(N, Cc, P, 1)
    got_dx = dx.cpu().double().permute(0, 2, 1).reshape(N, Cc, P, 1)
    tol = 1.0 / 128 if precision == "bf16" else 2e-5
    ey = ((got_y - yr.detach()).abs() * sure).max().item() / yr.abs().max().item()
    edx = ((got_dx - dxr).abs() * sure).max().item() / dxr.abs().max().item()
    mean_ref = x.double().reshape(N, P, 32, Cc // 32).mean((1, 3))
    rstd_ref = 1.0 / torch.sqrt(x.double().reshape(N, P, 32, Cc // 32).var((1, 3), unbiased=False) + 1e-5)
    assert (stats[:, :, 0].cpu().double() - mean_ref).abs().max().item() <= 1e-4
    # the statistics-only pass (streaming kernel in front of the tcgen05 GEMM / the classifier head): same (mean, rstd)
    stats2 = torch.full((N, 32, 2), float("nan"), device=DEV)
    _lib.check(e.lib.dp_debug_gn(e.handle, _ptr(xd), None, None, _ptr(gd), _ptr(bd), 1, None, None, _ptr(stats2), N, P, Cc, e._stream()))
    torch.cuda.synchronize()
    assert (stats2[:, :, 0].cpu().double() - mean_ref).abs().max().item() <= 1e-4
    assert ((stats2[:, :, 1].cpu().double() - rstd_ref).abs() / rstd_ref).max().item() <= 1e-4
    assert ((stats[:, :, 1].cpu().double() - rstd_ref).abs() / rstd_ref).max().item() <= 1e-4
    print(precision, P, Cc, "neg" if neg_gamma else "", "rel err y %.2e dx %.2e" % (ey, edx))
    assert ey <= tol and edx <= tol, (ey, edx)


# (B, S, samples per launch): one launch over the whole step, and launch sequences that split images as the chunk loop does
STEM_BWD_LAUNCHES = [(2, 3, 6), (1, 5, 5), (2, 5, 4), (3, 3, 2), (1, 7, 7)]


@pytest.mark.parametrize("B,S,step", STEM_BWD_LAUNCHES)
def test_bf16_stem_bwd_reduce_vs_torch_fp32(engines, oracle_params, B, S, step):
    """The K1^T the bf16 bench runs: G[b] = 2 * sum_s keep_{b,s} * conv7x7s2^T(dY_{b,s}, W) with W the standardised stem
    weights as the engine holds them (bf16), dY bf16 -- against torch fp32 conv_transpose2d on the same bf16-rounded
    operands (the factor 2 is d((x-0.5)/0.5)/dx, utils.py:77-78; keep = attack.py:206).  Both sides multiply exact
    bf16 products and accumulate in fp32; only the summation order differs: relative L2 <= 1e-5, max abs <= 1e-4 of max.
    The samples run in launches of `step` (dp_debug_k1t, samples [n0, n0 + step)) into a G that starts as NaN: the
    launch holding an image's first sample must overwrite it, later launches add.  The split sequences also hold one
    fully occluded sample."""
    from dorpatch_b200 import _lib, masks as PM
    e = engines("bf16")
    H, hs = 224, 112
    N = B * S
    dY = (_rand((N, hs, hs, 64), 11, 1.0) * 1e-2).to(torch.bfloat16)
    idx = np.random.RandomState(7).randint(0, 2520, (B, S))
    rects = PM.gather(PM.universe(H, 2), idx)
    rects_c = np.ascontiguousarray(rects.reshape(N, 4, 4), np.int16)
    keep = torch.from_numpy(OM.rects_to_bool(OM.universe_rects(H, 2), H))[torch.as_tensor(idx.reshape(-1))].float()
    if step < N or N == 7:
        rects_c[1] = 0
        rects_c[1, 0] = (0, H, 0, H)
        keep[1] = 0.0
    G = torch.full((B, 3, H, H), float("nan"), device=DEV)
    dYd = dY.to(DEV)
    for n0 in range(0, N, step):
        n = min(step, N - n0)
        _lib.check(e.lib.dp_debug_k1t(e.handle, _ptr(dYd[n0:n0 + n]), C.c_void_p(rects_c.ctypes.data), B, S, n0, n, _ptr(G),
                                      e._stream()))
    torch.cuda.synchronize()
    w = OR.standardize(oracle_params["stem.conv.weight"]).to(torch.bfloat16).float()         # [64,3,7,7]
    dX = F.conv_transpose2d(dY.float().permute(0, 3, 1, 2), w, stride=2, padding=3, output_padding=1)   # [N,3,224,224]
    ref = 2.0 * (dX * keep).reshape(B, S, 3, H, H).sum(1)
    got = G.cpu()
    assert torch.isfinite(got).all()
    rel = float((got - ref).norm() / ref.norm())
    mx = float((got - ref).abs().max() / ref.abs().max())
    print("stem_bwd_reduce B=%d S=%d launches of %d vs torch fp32: rel L2 %.2e, max abs / max %.2e" % (B, S, step, rel, mx))
    assert rel <= 1e-5 and mx <= 1e-4, (rel, mx)


GEMM_SHAPES = [  # (N, P, K, Nout, shortcut): conv3 of every stage (with the residual), conv1 shapes, ragged M
    (2, 3136, 64, 256, True), (3, 784, 128, 512, True), (5, 196, 256, 1024, True), (7, 49, 512, 2048, True),
    (2, 3136, 256, 64, False), (3, 784, 512, 128, False), (5, 196, 1024, 256, False), (3, 49, 2048, 512, False),
]


@pytest.mark.parametrize("N,P,K,Nout,shortcut", GEMM_SHAPES)
def test_tcgen05_gn_gemm_vs_fp32(engines, N, P, K, Nout, shortcut):
    """kernels_gemm.cu (tcgen05.mma, TMEM accumulators): out = relu(gn(x)) @ W^T (+ shortcut) with relu(gn(x)) rounded to
    bf16 on its way into shared memory, against the same product in torch fp32 on the same bf16-rounded operands
    (timm PreActBottleneck norm1->conv1 / norm3->conv3 + residual).  fp32 accumulation on both sides, output rounded to
    bf16: |diff| <= 1/128 of the output's max (one bf16 ulp at the top of the range) and relative L2 <= 4e-3."""
    from dorpatch_b200 import _lib
    e = engines("bf16")
    M = N * P
    x = _rand((N, P, K), 21, 1.5, 0.4).to(torch.bfloat16)
    w = (_rand((Nout, K), 22) / np.sqrt(K) * 2).to(torch.bfloat16)
    gamma, beta = 1.0 + 0.3 * _rand((K,), 23), 0.3 * _rand((K,), 24)
    r = _rand((M, Nout), 25).to(torch.bfloat16) if shortcut else None
    xf = x.float()
    cpg = K // 32
    grp = xf.reshape(N, P, 32, cpg)
    mean = grp.mean((1, 3))
    rstd = 1.0 / torch.sqrt(grp.var((1, 3), unbiased=False) + 1e-5)
    stats = torch.stack([mean, rstd], -1).contiguous()                                   # [N,32,2]
    sa = rstd.repeat_interleave(cpg, 1) * gamma[None]                                    # [N,K]
    sb = beta[None] - mean.repeat_interleave(cpg, 1) * sa
    yb = torch.relu(torch.addcmul(sb[:, None, :], sa[:, None, :], xf)).to(torch.bfloat16).float()   # fmaf(sa, x, sb) rounded to bf16
    ref = yb.reshape(M, K) @ w.float().t()
    if shortcut:
        ref = ref + r.float()
    out = torch.empty(M, Nout, dtype=torch.bfloat16, device=DEV)
    xd, wd, sd, gd, bd = x.to(DEV), w.to(DEV), stats.to(DEV), gamma.to(DEV), beta.to(DEV)     # keep the device copies alive
    rd = r.to(DEV) if shortcut else None
    _lib.check(e.lib.dp_debug_gn_gemm(e.handle, _ptr(xd), _ptr(wd), _ptr(sd), _ptr(gd), _ptr(bd), _ptr(rd), _ptr(out), N, P, K, Nout,
                                      e._stream()))
    torch.cuda.synchronize()
    got = out.cpu().float()
    assert torch.isfinite(got).all()
    mx = float((got - ref).abs().max() / ref.abs().max())
    rel = float((got - ref).norm() / ref.norm())
    print("gn_gemm N=%d P=%d K=%d Nout=%d: max abs / max %.2e, rel L2 %.2e" % (N, P, K, Nout, mx, rel))
    assert mx <= 1.0 / 128 and rel <= 4e-3, (mx, rel)


def test_device_failed_set_equals_host_state_machine(engines):
    """The failed-mask set kept as a device bitmap (dp_failed_set_write / _update / _read, SURVEY 8f N2) against the host
    list arithmetic of attack.py:259-267 (np.setdiff1d / np.unique) driven by the same sampler over 400 random steps of two
    images: identical set sizes every step, identical sorted contents whenever the sampler reads them, identical samples."""
    from dorpatch_b200.attack import _ImageState
    e = engines("fp32")
    B, S, n_mask = 2, 8, 2520
    host = [_ImageState(0.01, 1e-3, 3, False, np.random.RandomState(10 + b)) for b in range(B)]
    dev = [_ImageState(0.01, 1e-3, 3, False, np.random.RandomState(10 + b)) for b in range(B)]
    for b, s in enumerate(dev):
        s.dev = (e, b)
    rng = np.random.RandomState(0)
    for b in range(B):
        init = sorted(rng.choice(n_mask, 40, replace=False).tolist())
        host[b].failed, host[b].n_failed = list(init), len(init)
        dev[b].set_failed(init)
    for i in range(990, 1390):                       # crosses i == 1000, where half of the samples start to come from the set
        idx_h, idx_d, nff_h, nff_d = [], [], [], []
        for b in range(B):
            a, na = host[b].sample(i, n_mask, S)
            c, nc = dev[b].sample(i, n_mask, S)
            assert na == nc and np.array_equal(a, c)
            idx_h.append(a); nff_h.append(na); idx_d.append(c); nff_d.append(nc)
        loss = (rng.rand(B, S) < 0.6).astype(np.float32) * 0.5
        counts = e.failed_update(np.stack(idx_d), nff_d, [True] * B, loss=loss)
        for b in range(B):
            ra = host[b].bookkeeping(1, i, loss[b], idx_h[b], nff_h[b], 1.0)
            rb = dev[b].bookkeeping(1, i, loss[b], idx_d[b], nff_d[b], 1.0, n_failed=counts[b])
            assert ra == rb and host[b].n_failed == dev[b].n_failed == counts[b]
            assert (host[b].lr, host[b].structured, host[b].not_decay, host[b].num_failure) == (dev[b].lr, dev[b].structured, dev[b].not_decay, dev[b].num_failure)
        if i % 50 == 0:
            for b in range(B):
                assert e.failed_read(b) == host[b].failed
    inactive = e.failed_update(np.zeros((B, S), np.int32), [0] * B, [False] * B, loss=np.ones((B, S), np.float32))
    assert [int(v) for v in inactive] == [host[b].n_failed for b in range(B)]      # inactive images are left untouched
