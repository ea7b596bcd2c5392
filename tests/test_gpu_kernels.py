"""GPU parity tests: every native kernel / engine entry point (called through the C ABI)
against the CPU oracle on the same seeded inputs.  Tolerances are stated per test."""
import numpy as np
import pytest
import torch

from oracle import attack as OA
from oracle import masks as OM
from oracle import resnetv2 as OR

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rand(shape, seed):
    return torch.rand(shape, generator=torch.Generator().manual_seed(seed))


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a @ b) / (a.norm() * b.norm() + 1e-30))


def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))


def _rects_for(H, idx, dropout=2, idx2=None):
    table = OM.rects_to_array(OM.universe_rects(H, dropout))
    out = np.zeros(np.asarray(idx).shape + (4, 4), np.int16)
    out[..., 0:2, :] = table[np.asarray(idx)]
    if idx2 is not None:
        out[..., 2:4, :] = table[np.asarray(idx2)]
    return out


# --------------------------------------------------------------------------------------
@pytest.mark.parametrize("H", [56, 224])
def test_paste_matches_clip(engine_factory, H):
    """utils.clip + add.  fp32; tolerance 2e-6 abs (the L2 norm reduction order differs)."""
    e = engine_factory(img=H, precision="fp32", chunk=4, max_images=4)
    B = 3
    x, m, p = _rand((B, 3, H, H), 1), _rand((B, 1, H, H), 2), _rand((B, 3, H, H), 3)
    m[1] *= 0.01          # image 1: ||delta|| < eps -> scale exactly 1
    m[2] *= 0.0           # image 2: zero delta -> eps/0 = inf -> clipped to 1
    adv, l2, sc = e.paste(x.to(DEV), m.to(DEV), p.to(DEV), 4.0)
    torch.cuda.synchronize()
    ref = x + OA.clip_paste(m, p, x, 4.0)
    ref_l2 = torch.norm(m * (p - x), p=2, dim=(1, 2, 3))
    assert np.allclose(l2, ref_l2.numpy(), rtol=1e-5)
    assert sc[1] == 1.0 and sc[2] == 1.0 and sc[0] < 1.0
    assert (adv.cpu() - ref).abs().max().item() <= 2e-6


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("H,S", [(56, 5), (224, 7)])
def test_expand_matches_occlude_normalise(engine_factory, precision, H, S):
    """K1 (non-fused entry): (occlude(img) - 0.5)/0.5 in NHWC.  fp32: bit-exact;
    bf16: equal to the bf16 rounding of the fp32 result."""
    e = engine_factory(img=H, precision=precision, chunk=4, max_images=4)
    B = 2
    img = _rand((B, 3, H, H), 5)
    rng = np.random.RandomState(0)
    idx, idx2 = rng.randint(0, 2520, (B, S)), rng.randint(0, 2520, (B, S))
    idx[0, 0] = 0
    rects = _rects_for(H, idx, 2, idx2)
    rects[1, 1] = 0                                        # one sample without any occluder
    out = e.expand(img.to(DEV), S, rects)
    torch.cuda.synchronize()
    uni = torch.from_numpy(OM.rects_to_bool(OM.universe_rects(H, 2), H))
    ref = OA.occlude(OA.occlude(img[:, None], uni[idx.reshape(-1)].reshape(B, S, 1, H, H)),
                     uni[idx2.reshape(-1)].reshape(B, S, 1, H, H))
    ref[1, 1] = img[1]
    ref = ((ref - 0.5) / 0.5).reshape(B * S, 3, H, H).permute(0, 2, 3, 1)
    got = out.float().cpu()
    assert got.shape[-1] == e.c_pad
    assert (got[..., 3:] == 0).all()
    if precision == "fp32":
        assert torch.equal(got[..., :3], ref)
    else:
        assert torch.equal(got[..., :3], ref.bfloat16().float())


def _torch_gpu_reference(params, z, dl, precision):
    """The same network in PyTorch on the GPU at the given arithmetic: what the reference itself
    would compute on a GPU (its default is TF32 convolutions, utils.py:17 / torch defaults)."""
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = precision != "fp32"
    try:
        pg = {k: v.to(DEV) for k, v in params.items()}
        zc = z.to(DEV).requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(precision == "bf16")):
            out = OR.forward_normalized(pg, zc)
        (out.float() * dl.to(DEV)).sum().backward()
        return out.float().detach().cpu(), zc.grad.cpu()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.mark.parametrize("precision,tol_logit,min_cos", [("fp32", 2e-3, 0.999), ("tf32", None, None), ("bf16", None, None)])
def test_classifier_forward_backward(engine_factory, oracle_params, precision, tol_logit, min_cos):
    """ResNetV2-50 logits and d/d(input) vs torch-CPU autograd on the oracle restatement.
    fp32: |dlogit| <= 2e-3, grad cosine >= 0.999 (ReLU / max-pool ties flip on last-bit
    differences, so gradients are compared by cosine, not element-wise).
    tf32 / bf16: the random-init network is chaotic in its input gradient (PyTorch's own GPU
    run at the same arithmetic drifts from fp32-CPU by the same amount -- measured cos 0.94 /
    0.52), so the bar is "no further from the fp32 oracle than PyTorch-GPU at that arithmetic":
    logit error <= 2x PyTorch's + 5e-3, gradient cosine >= PyTorch's - 0.05."""
    H, N = 112, 3
    e = engine_factory(img=H, precision=precision, chunk=8, max_images=4)
    z = (_rand((N, 3, H, H), 11) - 0.5) * 2
    dl = torch.zeros(N, 1000)
    dl[torch.arange(N), torch.tensor([3, 500, 999])] = 1.0
    dl[torch.arange(N), torch.tensor([7, 1, 0])] = -1.0
    logits, dz = e.net_forward_backward(z.to(DEV), dl.to(DEV))
    torch.cuda.synchronize()
    zr = z.clone().requires_grad_(True)
    ref = OR.forward_normalized(oracle_params, zr)
    (ref * dl).sum().backward()
    err = (logits.cpu() - ref.detach()).abs().max().item()
    cos = _cos(dz.cpu(), zr.grad)
    print("precision", precision, "logit err", err, "grad cos", cos, "rel", _rel(dz.cpu(), zr.grad))
    if precision != "fp32":
        t_logits, t_grad = _torch_gpu_reference(oracle_params, z, dl, precision)
        t_err = (t_logits - ref.detach()).abs().max().item()
        t_cos = _cos(t_grad, zr.grad)
        print("  torch-GPU at", precision, ": logit err", t_err, "grad cos", t_cos)
        tol_logit, min_cos = 2 * t_err + 5e-3, t_cos - 0.05
    assert err <= tol_logit, err
    assert cos >= min_cos, cos


def test_predict_matches_oracle(engine_factory, oracle_net):
    """dp_predict (K1 + forward + argmax), fp32: logits within 2e-3 of the oracle and the
    same argmax wherever the oracle's top-2 margin exceeds 1e-2."""
    H, B, S = 112, 2, 5
    e = engine_factory(img=H, precision="fp32", chunk=8, max_images=4)
    img = _rand((B, 3, H, H), 21)
    idx = np.random.RandomState(1).randint(0, 144, (B, S))
    rects = _rects_for(H, idx, 1)
    preds, logits = e.predict(img.to(DEV), S, rects, return_logits=True)
    uni = torch.from_numpy(OM.rects_to_bool(OM.universe_rects(H, 1), H))
    with torch.no_grad():
        ref = oracle_net(OA.occlude(img[:, None], uni[idx.reshape(-1)].reshape(B, S, 1, H, H)).reshape(B * S, 3, H, H))
    assert np.abs(logits - ref.numpy()).max() <= 2e-3
    top2 = ref.topk(2, dim=1).values
    sure = (top2[:, 0] - top2[:, 1]) > 1e-2
    assert (torch.from_numpy(preds).long()[sure] == ref.argmax(1)[sure]).all()
    # no-occlusion path (model(x))
    p0 = e.predict(img.to(DEV))
    with torch.no_grad():
        r0 = oracle_net(img)
    t2 = r0.topk(2, dim=1).values
    s0 = (t2[:, 0] - t2[:, 1]) > 1e-2
    assert (torch.from_numpy(p0).long()[s0] == r0.argmax(1)[s0]).all()


@pytest.mark.parametrize("stage", [0, 1])
def test_attack_step_matches_oracle(engine_factory, oracle_net, stage):
    """One hot-loop iteration (attack.py:184-247 + :332-342), fp32 engine, B=2 x S=3, two
    chunks.  loss_adv / regularisers: 2e-3 abs (rel 1e-4 for the lasso); gradients:
    cosine >= 0.999 and sign agreement >= 99% where |g| is above 1e-3 of its max."""
    H, B, S = 112, 2, 3
    e = engine_factory(img=H, precision="fp32", chunk=4, max_images=4)
    x, m, p = _rand((B, 3, H, H), 31), _rand((B, 1, H, H), 32), _rand((B, 3, H, H), 33)
    if stage == 1:
        m = (m > 0.8).float()
    else:
        m[0, 0, :7, :7] = 0.0                      # an all-zero 7x7 group -> NaN grad -> frozen (quirk Q5)
    y = torch.tensor([17, 400])
    targeted = [True, False]
    idx = np.random.RandomState(3).randint(0, 2520, (B, S))
    rects = _rects_for(H, idx, 2)
    structured, coeff = [1e-3, 5e-4], [1e-5, 3e-5]
    density = 1e-3
    xd, md, pd = x.to(DEV), m.to(DEV).clone(), p.to(DEV).clone()
    G = torch.zeros(B, 3, H, H, device=DEV)
    r = e.attack_grad(xd, md, pd, rects, y.numpy(), targeted, 0.1, 4.0, stage, G)
    gp, gm = torch.zeros_like(pd), torch.zeros_like(md)
    lr = np.array([0.01, 0.02], np.float32)
    e.attack_update(xd, md, pd, G, lr, structured, coeff, density, stage, grad_pattern_out=gp, grad_mask_out=gm)
    torch.cuda.synchronize()

    uni = torch.from_numpy(OM.rects_to_bool(OM.universe_rects(H, 2), H))
    lvx = OA.local_variance(x)[0].mean(1)
    o = OA.step_losses_and_grads(oracle_net, x, m, p, y, idx, uni, targeted, 1000, 0.1, structured, density,
                                 coeff, stage, 4.0, lvx)
    print("loss_adv", r["loss_adv"], o["loss_adv"].numpy())
    assert np.abs(r["loss_adv"] - o["loss_adv"].numpy()).max() <= 2e-3
    assert np.allclose(r["loss_struc"], o["loss_struc"].numpy(), rtol=1e-4, atol=1e-6)
    top2 = o["logits"].topk(2, dim=1).values
    sure = ((top2[:, 0] - top2[:, 1]) > 1e-2).numpy()
    assert (r["preds"].reshape(-1)[sure] == o["logits"].argmax(1).numpy()[sure]).all()
    if stage == 0:
        assert np.allclose(r["loss_density"], o["loss_density"].numpy(), rtol=1e-4)
        assert np.allclose(r["group_lasso"], o["group_lasso"].numpy(), rtol=1e-4)

    def check_grad(name, got, ref):
        ref = torch.nan_to_num(ref, nan=0.0)
        got = torch.nan_to_num(got.cpu(), nan=0.0)
        cos = _cos(got, ref)
        big = ref.abs() > 1e-3 * ref.abs().max()
        agree = (got.sign()[big] == ref.sign()[big]).float().mean().item()
        print(name, "cos", cos, "sign agreement", agree)
        assert cos >= 0.999, (name, cos)
        assert agree >= 0.99, (name, agree)

    check_grad("grad_pattern", gp, o["grad_pattern"])
    # sign step
    pref = (p - torch.from_numpy(lr)[:, None, None, None] * torch.nan_to_num(gp.cpu()).sign()).clamp(0, 1)
    assert torch.equal(pd.cpu(), pref)
    if stage == 0:
        nan_ref = torch.isnan(o["grad_mask"])
        assert nan_ref[0, 0, :7, :7].all()
        assert torch.isnan(gm.cpu())[nan_ref].all()                       # NaN reproduced ...
        assert torch.equal(md.cpu()[nan_ref], m[nan_ref])                 # ... and those pixels frozen
        check_grad("grad_mask", gm, o["grad_mask"])
        mref = (m - torch.from_numpy(lr)[:, None, None, None] * torch.nan_to_num(gm.cpu()).sign()).clamp(0, 1)
        assert torch.equal(md.cpu(), mref)
    else:
        assert torch.equal(md.cpu(), m)


def test_window_sum(engine_factory):
    H = 112
    e = engine_factory(img=H, precision="fp32", chunk=8, max_images=4)
    m = _rand((2, 1, H, H), 41)
    got = e.window_sum(m.to(DEV), 7)
    ref = OA.window_sum(m, 7).reshape(2, -1).numpy()
    assert np.allclose(got, ref, rtol=1e-5)


def test_affine_colour_eot_step_matches_torch_oracle(engine_factory, oracle_net):
    """Optional affine / colour EOT (not in the reference; oracle = F.affine_grid/grid_sample):
    one step with per-sample transforms, fp32 engine.  loss 2e-3 abs; grad cosine >= 0.999."""
    from dorpatch_b200 import eot as PE
    H, B, S = 112, 2, 3
    e = engine_factory(img=H, precision="fp32", chunk=4, max_images=4)
    x, m, p = _rand((B, 3, H, H), 51), _rand((B, 1, H, H), 52), _rand((B, 3, H, H), 53)
    y = torch.tensor([17, 400])
    targeted = [True, False]
    idx = np.random.RandomState(4).randint(0, 2520, (B, S))
    rects = _rects_for(H, idx, 2)
    xf = PE.sample(np.random.RandomState(9), B, S, affine=1.0, colour=1.0)
    xf[0, 0] = [1, 0, 0, 0, 1, 0, 1, 0]                              # identity transform on one sample
    G = torch.zeros(B, 3, H, H, device=DEV)
    xd, md, pd = x.to(DEV), m.to(DEV).clone(), p.to(DEV).clone()
    r = e.attack_grad(xd, md, pd, rects, y.numpy(), targeted, 0.1, 4.0, 1, G, xforms=xf)
    gp = torch.zeros_like(pd)
    e.attack_update(xd, md, pd, G, np.zeros(B, np.float32), [0.0, 0.0], None, 0.0, 1, grad_pattern_out=gp)
    torch.cuda.synchronize()
    uni = torch.from_numpy(OM.rects_to_bool(OM.universe_rects(H, 2), H))
    o = OA.step_losses_and_grads(oracle_net, x, m, p, y, idx, uni, targeted, 1000, 0.1, [0.0, 0.0], 0.0, [0.0, 0.0], 1,
                                 4.0, OA.local_variance(x)[0].mean(1), xforms=xf)
    print("eot loss", r["loss_adv"], o["loss_adv"].numpy())
    assert np.abs(r["loss_adv"] - o["loss_adv"].numpy()).max() <= 2e-3
    cos = _cos(gp.cpu(), o["grad_pattern"])
    print("eot grad cos", cos)
    assert cos >= 0.999, cos


def test_reference_named_helpers_on_gpu(oracle_params):
    """utils.clip / DorPatch.patch_selection / DorPatch.collect_failure keep the reference's signatures
    and semantics (utils.py:105-110, attack.py:363-406) on the native engine."""
    import os
    from dorpatch_b200 import masks as PM
    from dorpatch_b200.attack import DorPatch
    from dorpatch_b200.resnetv2 import ResNetV2
    from dorpatch_b200.utils import NormModel, clip, get_normalize
    os.environ["DORPATCH_PRECISION"] = "fp32"
    os.environ["DORPATCH_CHUNK"] = "16"
    H = 112
    x, m, p = _rand((2, 3, H, H), 61), _rand((2, 1, H, H), 62), _rand((2, 3, H, H), 63)
    d = clip(m.to(DEV), p.to(DEV), x.to(DEV), 4.0)
    assert (d.cpu() - OA.clip_paste(m, p, x, 4.0)).abs().max().item() <= 1e-6
    sel = DorPatch().patch_selection(m.to(DEV), 0.10)
    assert torch.equal(sel.cpu(), OA.patch_selection(m, 0.10))
    net = ResNetV2(seed=0)
    net.load_state_dict(oracle_params)
    model = torch.nn.DataParallel(NormModel(net, get_normalize("imagenet", "resnetv2"))).cuda().eval()
    onet = OR.OracleNet(oracle_params, weights_require_grad=False).eval()
    uni = torch.from_numpy(OM.rects_to_bool(OM.universe_rects(H, 1), H))
    with torch.no_grad():
        logits = onet(OA.occlude(x[:1], uni))
    y = int(logits.argmax(1).mode()[0])
    ref_failed = OA.collect_failure(onet, x[:1], y, uni, False, 64)
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        got = DorPatch().collect_failure(x[:1].to(DEV), torch.tensor([y]), PM.universe(H, 1), False, model, batch_size=64)
        got_bool = DorPatch().collect_failure(x[:1].to(DEV), torch.tensor([y] * 64).to(DEV), uni.to(DEV), False, model, batch_size=64)
    top2 = logits.topk(2, dim=1).values
    unsure = set(np.nonzero(((top2[:, 0] - top2[:, 1]) < 1e-3).numpy())[0].tolist())
    assert set(got) ^ set(ref_failed) <= unsure
    assert set(got_bool) ^ set(ref_failed) <= unsure


def test_bf16_fused_stem_backward_reduce_matches_library_path(oracle_params):
    """bf16 engine: the hand-written stem dgrad fused with the masked EOT reduce (no per-sample input
    gradient tensor) against the same engine using cuDNN's stem dgrad + reduce_kernel.  Same bf16
    inputs; the library path additionally rounds every sample's input gradient to bf16 before the
    reduce, so: cosine >= 0.9999, relative L2 error <= 1e-2; losses identical."""
    import os
    from dorpatch_b200.engine import Engine
    H, B, S = 112, 2, 5
    x, m, p = _rand((B, 3, H, H), 71), _rand((B, 1, H, H), 72), _rand((B, 3, H, H), 73)
    idx = np.random.RandomState(5).randint(0, 2520, (B, S))
    rects = _rects_for(H, idx, 2)
    y = np.array([17, 400])
    out = {}
    for mode in ("fused", "cudnn"):
        os.environ["DORPATCH_STEM_BWD"] = mode
        e = Engine(img=H, precision="bf16", chunk=4, max_images=B, autotune=False)   # 3 chunks: images straddle chunks
        e.load_state_dict(oracle_params)
        G = torch.zeros(B, 3, H, H, device=DEV)
        r = e.attack_grad(x.to(DEV), m.to(DEV), p.to(DEV), rects, y, [True, False], 0.1, 4.0, 1, G)
        torch.cuda.synchronize()
        out[mode] = (G.cpu().clone(), r["loss_adv"].copy())
        e.close()
    os.environ.pop("DORPATCH_STEM_BWD", None)
    assert np.array_equal(out["fused"][1], out["cudnn"][1])
    cos, rel = _cos(out["fused"][0], out["cudnn"][0]), _rel(out["fused"][0], out["cudnn"][0])
    print("fused stem bwd vs library: cos", cos, "rel", rel)
    assert cos >= 0.9999 and rel <= 1e-2, (cos, rel)


# engine option (read at create) -> (its two settings, B, S): results must not depend on it
ENGINE_OPTIONS = {
    # dp_attack_grad alternates chunks between two workspaces / streams when every chunk holds whole images
    # (chunk 4, S 4: 3 chunks of one image each on lanes 0, 1, 0)
    "DORPATCH_LANES": (("1", "2"), 3, 4),
    # K1 per classifier chunk (0: launches [n0, n0+4) that split the 3-sample images) against one whole-step launch
    "DORPATCH_K1_WHOLE_MB": (("0", None), 3, 3),
}


@pytest.mark.parametrize("option", list(ENGINE_OPTIONS))
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_engine_option_does_not_change_results(oracle_params, precision, option):
    """Same kernels, same inputs, a different schedule: one dp_attack_grad step must give the same patch gradient,
    per-sample losses and predictions bit for bit under either setting of the option (None = unset, the default)."""
    import os
    from dorpatch_b200.engine import Engine
    settings, B, S = ENGINE_OPTIONS[option]
    H = 112
    x, m, p = _rand((B, 3, H, H), 81), _rand((B, 1, H, H), 82), _rand((B, 3, H, H), 83)
    rects = _rects_for(H, np.random.RandomState(6).randint(0, 2520, (B, S)), 2)
    y = np.array([1, 2, 3])
    out = {}
    for value in settings:
        if value is None:
            os.environ.pop(option, None)
        else:
            os.environ[option] = value
        try:
            e = Engine(img=H, precision=precision, chunk=4, max_images=B, autotune=False)
        finally:
            os.environ.pop(option, None)
        e.load_state_dict(oracle_params)
        G = torch.full((B, 3, H, H), float("nan"), device=DEV)
        r = e.attack_grad(x.to(DEV), m.to(DEV), p.to(DEV), rects, y, [True, False, True], 0.1, 4.0, 0, G)
        torch.cuda.synchronize()
        out[value] = (G.cpu().clone(), r["loss_adv"].copy(), r["preds"].copy())
        e.close()
    a, b = (out[v] for v in settings)
    assert torch.isfinite(a[0]).all()
    assert torch.equal(a[0], b[0])
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_cuda_graph_replay_is_bit_identical(oracle_params, precision):
    """dp_attack_grad captures its launch sequence into a CUDA graph on the second call of a signature and replays it
    afterwards (SURVEY 8f N4).  Same kernels, same order, fresh staging contents per call: every call must equal the
    eager engine (DORPATCH_GRAPH=0) bit for bit, including calls whose rectangles / labels differ from the captured one."""
    import os
    from dorpatch_b200.engine import Engine
    H, B, S = 112, 3, 4                       # chunk 4 -> 3 chunks on two lanes
    x, m, p = _rand((B, 3, H, H), 91), _rand((B, 1, H, H), 92), _rand((B, 3, H, H), 93)
    calls = [(_rects_for(H, np.random.RandomState(10 + k).randint(0, 2520, (B, S)), 2), np.array([1 + k, 2, 3 + 5 * k])) for k in range(4)]
    out = {}
    for graph in ("0", "1"):
        os.environ["DORPATCH_GRAPH"] = graph
        e = Engine(img=H, precision=precision, chunk=4, max_images=B, autotune=False)
        e.load_state_dict(oracle_params)
        xd, md, pd = x.to(DEV), m.to(DEV), p.to(DEV)
        G = torch.zeros(B, 3, H, H, device=DEV)
        res = []
        for rects, y in calls:
            r = e.attack_grad(xd, md, pd, rects, y, [True, False, True], 0.1, 4.0, 0, G)
            torch.cuda.synchronize()
            res.append((G.cpu().clone(), r["loss_adv"].copy(), r["preds"].copy(), r["group_lasso"].copy()))
        out[graph] = res
        replays, why = e.graph_replays, e.graph_status
        e.close()
        assert replays == (3 if graph == "1" else 0), (replays, why)        # call 1 eager, call 2 capture + launch, calls 3-4 replay
    os.environ.pop("DORPATCH_GRAPH", None)
    for a, b in zip(out["0"], out["1"]):
        assert torch.equal(a[0], b[0])
        assert all(np.array_equal(u, v) for u, v in zip(a[1:], b[1:]))
