#!/usr/bin/env python
"""bench.py -- EOT-samples/sec of the DorPatch hot loop (BASELINE.json metric).

    python bench.py [--gpus N --steps K --warmup W] [--impl native|reference] [--precision tf32|bf16|fp32] [--dump-outputs DIR]

A "step" is one iteration of attack.py:184-342 of the reference over one batch: sample occlusion masks on the host,
paste + expand (K1), ResNetV2-50x1-BiT forward + backward-to-input (K2), CW loss (K4), masked EOT gradient reduce
(K1^T), [all-reduce across ranks], host bookkeeping, sign step (K3).

HEADLINE workload = BASELINE.json configs[2] ("c3", the largest single-GPU configuration): 64 synthetic 224x224 images
x 32 EOT double-mask occlusion samples (dropout=2, the 2520-mask universe), stage-1 step, at the REFERENCE'S OWN GPU
ARITHMETIC: fp32 storage, TF32 tensor-core convolutions (`--precision tf32`; PyTorch's cudnn.allow_tf32 default that
the reference runs with).  Weak scaling keeps 2048 EOT samples per GPU and step: N=1 64x32, N=2 64x64, N=4 128x64,
N=8 256x64 = configs[3] ("c4"); every rank holds all images and evaluates its slice of the EOT samples (one
all-reduce of the patch gradient per step).

Prints ONE JSON line (rank 0).  `value` = device-resident throughput, `e2e` = the same step through host buffers
(H2D of x/mask/pattern + D2H of mask/pattern/losses every step, dp_attack_step_host), `roofline` = the hand-written K1
kernel, timed on the variant and launch shape the step itself uses (one launch per step), against the measured HBM copy
bandwidth: `frac` counts the algorithmic bytes (3 channels), `frac_physical` the bytes really moved (the fp32 / tf32 network
input carries a zero pad channel for the library stem), `traffic` the DRAM bytes of that launch from the last ncu capture
(profiles/k1_traffic.json); `kernels` = per-category device time / achieved byte and flop rates of one profiled step,
`host_ms_per_step` = host time the GPU waits for, `graph_replays` = CUDA-graph replays of dp_attack_grad so far,
`cpu_baseline` = the oracle port of the reference's step on this box's host cores.  Extra legs (N=1 only; `legs`): the same step at bf16, configs[1] ("c2",
32 x 16) at both precisions, the reference's default shape (1 image x 128 EOT), the stage-0 step of configs[4]
("c5": targeted, 10 % budget, density + group-lasso regularisers live), PatchCleanser evaluation throughput, and the
scan-amortised throughput (the reference re-scans the whole mask universe every 100 steps, attack.py:187-190); the c3 / c2
legs carry the K1 roofline of their own launch shape (`k1_roofline`).  `--config c5s0 --gpus 4` = configs[4] on 4 GPUs.
Every timed run (headline, e2e, each leg) is K steps.

`--dump-outputs DIR` writes, after the headline's timed steps, what its last step handed back to the caller as DIR/<name>.npy
(float32): attack_grad's host results (loss_adv, preds, loss_struc, loss_density, group_lasso, l2), the patch gradient
grad_adv and the mask / pattern after the sign step.  An array of more than DUMP_MAX_ELEMENTS elements is written as the
same seeded sample of that many of its flattened elements (sorted indices), so the dump stays under 64 MB.  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMG = 224
SAMPLES_PER_GPU = 2048           # c3: 64 x 32
GFLOP_PER_SAMPLE = 16.36         # 8.18 fwd + 8.18 dgrad (SURVEY.md section 8d)
METRIC, UNIT = "EOT-samples/sec", "samples/s"
DUMP_MAX_ELEMENTS = 1 << 22
CONFIGS = {   # name -> (images, EOT per image [total], stage, targeted, budget)
    "c3": dict(B=64, S=32, stage=1, targeted=False, budget=0.12),
    "c2": dict(B=32, S=16, stage=1, targeted=False, budget=0.05),
    "b1": dict(B=1, S=128, stage=1, targeted=False, budget=0.12),      # the reference's defaults (main.py:27, attack.py:52-53)
    "c5s0": dict(B=32, S=16, stage=0, targeted=True, budget=0.10),     # configs[4] per-GPU share, stage-0 step
}


def shape_for(config, world):
    c = dict(CONFIGS[config])
    if config == "c3" and world > 1:              # weak scaling towards c4 (256 x 64 on 8 GPUs)
        c["S"] = 64
        c["B"] = SAMPLES_PER_GPU * world // 64
    elif world > 1:
        c["S"] = c["S"] * world
    return c


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k].startswith("Active") for r in self.rows)]
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(sm))


# ----------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's step on host cores
# ----------------------------------------------------------------------------------------------
def cpu_step_factory(S):
    import torch
    from oracle import attack as OA, masks as OM, resnetv2 as OR
    params = OR.random_init(seed=0)
    # "all the host threads it can use": torch-CPU convolutions on a small batch get SLOWER when oversubscribed
    # (128 threads: 0.14 samples/s on the GPU box), so pick the fastest thread count.
    cores = os.cpu_count() or 1
    cand = sorted({c for c in (8, 16, 32, 64, cores) if c <= min(cores, 64)})
    zt = torch.rand(4, 3, IMG, IMG).requires_grad_(True)
    best_t, best_dt = cand[0], float("inf")
    for c in cand:
        torch.set_num_threads(c)
        pr = {k: v.clone().requires_grad_(True) for k, v in params.items()}
        t0 = time.perf_counter()
        OR.forward(pr, zt).sum().backward()
        dt = time.perf_counter() - t0
        if dt < best_dt:
            best_t, best_dt = c, dt
        if dt > 4 * best_dt:
            break
    torch.set_num_threads(best_t)
    net = OR.OracleNet(params, weights_require_grad=True).eval()     # the reference never freezes the weights (Q7)
    g = torch.Generator().manual_seed(0)
    x = torch.rand(1, 3, IMG, IMG, generator=g)
    pattern = torch.rand(1, 3, IMG, IMG, generator=g)
    imp = torch.rand(1, 1, IMG, IMG, generator=g)
    mask = OA.patch_selection(imp, CONFIGS["c3"]["budget"])
    uni = torch.from_numpy(OM.rects_to_bool(OM.universe_rects(IMG, 2), IMG))
    lvx = OA.local_variance(x)[0].mean(1)
    with torch.no_grad():
        y = net(x).argmax(-1)
    rng = np.random.RandomState(0)
    state = dict(pattern=pattern)

    def step():
        idx = rng.choice(np.arange(uni.shape[0]), S, replace=False)[None]
        r = OA.step_losses_and_grads(net, x, mask, state["pattern"], y, idx, uni, [False], 1000, 0.1, [1e-3], 1e-3,
                                     [1e-5], 1, 4.0, lvx)
        state["pattern"] = (state["pattern"] - 0.01 * r["grad_pattern"].sign()).clamp(0, 1)
        return S
    return step, torch.get_num_threads()


def dump_outputs(arrays, out_dir):
    """arrays: name -> host array; written as float32 .npy files, larger ones as a fixed seeded sample (module docstring)."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, np.float32)
        if a.size > DUMP_MAX_ELEMENTS:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMENTS, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        total += a.nbytes
    assert total <= 64 << 20, total


def workload_config(config, world, precision=None):
    c = shape_for(config, world)
    name = {"c3": "configs[2] (c3)" if world == 1 else "c3 weak-scaled towards configs[3] (c4 = 256 x 64 on 8 GPUs)",
            "c2": "configs[1] (c2)", "b1": "reference default shape", "c5s0": "configs[4] (c5) per-GPU share, stage-0 step"}[config]
    return {"workload": "%s: batch %d x %d EOT (%d samples per GPU and step), 224x224, ResNetV2-50x1-BiT random-init, %d%% patch budget, "
                        "%s, stage-%d step, double-mask universe (2520)" % (name, c["B"], c["S"], c["B"] * c["S"] // world, round(c["budget"] * 100),
                                                                             "targeted" if c["targeted"] else "untargeted", c["stage"]),
            "images": c["B"], "eot_per_image_total": c["S"], "eot_per_image_per_gpu": c["S"] // world, "img": IMG,
            "parallelism": "eot-shard x%d + 1 allreduce(patch grad)/step" % world,
            "l2_policy": "inputs larger than L2 (>= 0.6 GB network input + tens of GB of activations per step)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    S = CONFIGS[args.config]["S"]
    step, threads = cpu_step_factory(S)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    n = 0
    for _ in range(args.steps):
        n += step()
    dt = time.perf_counter() - t0
    v = n / dt
    sample = ("1 image x %d EOT occlusion samples per step (same per-image work as the native arm; B scaled to 1 -- the reference is "
              "batch-size-1 only), stage-1 step, fp32, weights requires_grad as the reference" % S)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.config, args.gpus),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------------------------
class Workload:
    """One bench configuration on one engine: device-resident state, the host state machine, step / step_e2e."""

    def __init__(self, eng, config, world, rank, dev, dist):
        import torch
        from dorpatch_b200 import masks as PM
        from dorpatch_b200.attack import DorPatch, _ImageState
        c = shape_for(config, world)
        self.eng, self.world, self.rank, self.dev, self.dist = eng, world, rank, dev, dist
        self.B, self.S, self.S_loc, self.stage = c["B"], c["S"], c["S"] // world, c["stage"]
        B = self.B
        g = torch.Generator().manual_seed(1234)
        self.x = torch.rand(B, 3, IMG, IMG, generator=g).to(dev)
        self.pattern = torch.rand(B, 3, IMG, IMG, generator=g).to(dev)
        importance = torch.rand(B, 1, IMG, IMG, generator=g).to(dev)
        # stage 1: budget-sized binary mask from patch_selection; stage 0: the soft importance map itself is learnable
        self.mask = DorPatch().patch_selection(importance, c["budget"]) if self.stage == 1 else importance
        self.G = torch.zeros_like(self.x)
        self.table = PM.universe(IMG, 2)
        self.n_mask = self.table.shape[0]
        y = eng.predict(self.x).astype(np.int64)
        if c["targeted"]:
            y = (y + 1 + np.random.RandomState(5).randint(0, 998, B)) % 1000        # a target != the clean label
        self.y, self.crit = y, [bool(c["targeted"])] * B
        self.states = [_ImageState(0.01, 1e-3, y[b], c["targeted"], np.random.RandomState(1234 + b)) for b in range(B)]
        self.PM = PM
        self.nff0, self.act1 = np.zeros(B, np.int32), np.ones(B, np.uint8)
        self.host_s = 0.0
        from concurrent.futures import ThreadPoolExecutor
        self._pool, self._pref = ThreadPoolExecutor(max_workers=1), None
        self.hx = torch.empty(self.x.shape, pin_memory=True).copy_(self.x)
        self.hm = torch.empty(self.mask.shape, pin_memory=True).copy_(self.mask)
        self.hp = torch.empty(self.pattern.shape, pin_memory=True).copy_(self.pattern)
        if world > 1:
            self.dx, self.dm, self.dp_ = torch.empty_like(self.x), torch.empty_like(self.mask), torch.empty_like(self.pattern)

    @property
    def samples_per_step(self):
        return self.B * self.S

    def host_sample(self, i):
        idx = np.stack([s.sample(i, self.n_mask, self.S)[0] for s in self.states])
        return idx, self.PM.gather(self.table, idx[:, self.rank * self.S_loc:(self.rank + 1) * self.S_loc])

    def finish(self, i, idx, r, G):
        import torch
        loss_adv, work = r["loss_adv"], None
        if self.world > 1:
            from dorpatch_b200.attack import exchange_shards
            loss_adv, _, work = exchange_shards(self.dist, G, loss_adv, r["preds"], defer=True)   # all-reduce under the bookkeeping
        target = r["group_lasso"] if self.stage == 0 else r["loss_struc"]
        st_used = [s.structured for s in self.states]
        cg_used = [s.coeff_group_lasso for s in self.states]
        # failed-mask sets live on the device (as in DorPatch.generate): one kernel, the host reads the set sizes
        counts = self.eng.failed_update(idx, self.nff0, self.act1, loss=loss_adv if self.world > 1 else None)
        for b, s in enumerate(self.states):
            s.bookkeeping(self.stage, i, loss_adv[b], idx[b], 0, target[b], n_failed=counts[b])
        if work is not None:
            work.wait()                                   # orders the sign step after the all-reduce (stream dependency, no host block)
        return np.full(self.B, 0.01, np.float32), st_used, cg_used

    def _samples(self, i):
        # as DorPatch.generate: step i+1's indices are drawn on a helper thread while the GPU runs step i (i < 1000: the draw
        # depends on the per-image RNG streams only)
        if self._pref is not None and self._pref[0] == i:
            out = self._pref[1].result()
        else:
            out = self.host_sample(i)
        self._pref = (i + 1, self._pool.submit(self.host_sample, i + 1))
        return out

    def step(self, i):
        t0 = time.perf_counter()
        idx, rects = self._samples(i)
        self.host_s += time.perf_counter() - t0               # host time the GPU waits for (sampling that was not ready, rectangle gather)
        r = self.eng.attack_grad(self.x, self.mask, self.pattern, rects, self.y, self.crit, 0.1, 4.0, self.stage, self.G, S_total=self.S)
        t0 = time.perf_counter()
        lr, st_used, cg_used = self.finish(i, idx, r, self.G)
        self.host_s += time.perf_counter() - t0               # exchange + bookkeeping (the all-reduce runs under it)
        self.eng.attack_update(self.x, self.mask, self.pattern, self.G, lr, st_used, cg_used, 1e-3, self.stage)
        self.last = r

    def outputs(self):
        """What the last step() handed back: attack_grad's host results, the patch gradient, the updated mask / pattern."""
        out = {k: np.asarray(v, np.float32) for k, v in self.last.items()}
        out.update(grad_adv=self.G.cpu().numpy(), mask=self.mask.cpu().numpy(), pattern=self.pattern.cpu().numpy())
        return out

    def step_e2e(self, i):
        import torch
        idx, rects = self._samples(i)
        if self.world == 1:
            lr = np.full(self.B, 0.01, np.float32)
            st_used = [s.structured for s in self.states]
            cg_used = [s.coeff_group_lasso for s in self.states]
            r = self.eng.attack_step_host(self.hx.numpy(), self.hm.numpy(), self.hp.numpy(), rects, self.y, self.crit, 0.1, 4.0,
                                          self.stage, lr, st_used, cg_used, 1e-3, S_total=self.S)
            target = r["group_lasso"] if self.stage == 0 else r["loss_struc"]
            counts = self.eng.failed_update(idx, self.nff0, self.act1)
            for b, s in enumerate(self.states):
                s.bookkeeping(self.stage, i, r["loss_adv"][b], idx[b], 0, target[b], n_failed=counts[b])
        else:
            self.dx.copy_(self.hx, non_blocking=True); self.dm.copy_(self.hm, non_blocking=True); self.dp_.copy_(self.hp, non_blocking=True)
            r = self.eng.attack_grad(self.dx, self.dm, self.dp_, rects, self.y, self.crit, 0.1, 4.0, self.stage, self.G, S_total=self.S)
            lr, st_used, cg_used = self.finish(i, idx, r, self.G)
            self.eng.attack_update(self.dx, self.dm, self.dp_, self.G, lr, st_used, cg_used, 1e-3, self.stage)
            self.hm.copy_(self.dm, non_blocking=True); self.hp.copy_(self.dp_, non_blocking=True)
            torch.cuda.synchronize()

    def io_bytes(self):
        B, S = self.B, self.S_loc
        h2d = B * 7 * IMG * IMG * 4 + B * S * 32 + B * S * 5
        d2h = B * 4 * IMG * IMG * 4 + B * S * 8 + B * 16
        return int(h2d), int(d2h)


def run_native(args):
    import torch
    import torch.distributed as dist
    from dorpatch_b200.engine import Engine
    from dorpatch_b200.resnetv2 import ResNetV2

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl native needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, (world, args.gpus)
    pk = peaks()
    net = ResNetV2(seed=0)
    sd = net.state_dict()
    engines = {}

    def engine(precision):
        if precision not in engines:
            for e in engines.values():                  # one engine's workspace at a time
                e.close()
            engines.clear()
            e = Engine(img=IMG, precision=precision, chunk=args.chunk, max_images=max(shape_for(args.config, world)["B"], 64),
                       device=local, autotune=True)
            e.load_state_dict(sd)
            engines[precision] = e
        return engines[precision]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(eng, fn, K, i0):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = eng.launch_count
        e0.record()
        for k in range(K):
            fn(i0 + k)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), eng.launch_count - l0

    W, K = max(args.warmup, 3), args.steps

    def measure(precision, config, K, e2e=True, sampler=None, keep_outputs=False):
        eng = engine(precision)
        wl = Workload(eng, config, world, rank, dev, dist if world > 1 else None)
        for i in range(W):
            wl.step(i)
        if sampler is not None:
            sampler.start()
            time.sleep(0.3)
        wl.host_s = 0.0
        ms, launches = timed(eng, wl.step, K, W)
        clocks = sampler.stop() if sampler is not None else None
        outputs = wl.outputs() if keep_outputs else None
        res = dict(outputs=outputs, value=wl.samples_per_step * K / (ms / 1e3), ms_per_step=ms / K, launches=int(launches), clocks=clocks, wl=wl, eng=eng,
                   host_ms=wl.host_s / K * 1e3, graph_replays=eng.graph_replays)
        if e2e:
            for i in range(2):
                wl.step_e2e(W + K + i)
            ms_e2e, _ = timed(eng, wl.step_e2e, K, W + K + 2)
            res["e2e_value"] = wl.samples_per_step * K / (ms_e2e / 1e3)
            res["e2e_ms"] = ms_e2e / K
        return res

    if args.ncu:       # W warm-up steps, then ONE step inside cudaProfilerStart/Stop (for `ncu --profile-from-start off`)
        eng = engine(args.precision)
        wl = Workload(eng, args.config, world, rank, dev, None)
        for i in range(W):
            wl.step(i)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        wl.step(W)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return

    head = measure(args.precision, args.config, K, e2e=True, sampler=ClockSampler(local), keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(head.pop("outputs"), args.dump_outputs)
    wl, eng = head["wl"], head["eng"]
    h2d, d2h = wl.io_bytes()
    out = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.precision, "data": "synthetic", "config": workload_config(args.config, world),
        "clocks": head["clocks"], "gpu_launches": head["launches"],
        "host_ms_per_step": head["host_ms"], "graph_replays": head["graph_replays"],
        "e2e": {"value": head["e2e_value"], "unit": UNIT, "ms_per_step": head["e2e_ms"], "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h,
                "path": "dp_attack_step_host (C ABI, host buffers)" if world == 1 else "pinned host -> H2D -> grad/allreduce/update -> D2H"},
        "engine": {"chunk": args.chunk, "c_pad": eng.c_pad, "device_bytes": eng.device_bytes,
                   "gn": os.environ.get("DORPATCH_GN", "v2"), "fused_gemm": os.environ.get("DORPATCH_FUSED_GEMM", "0")},
        "precision_note": "tf32 = fp32 storage + TF32 tensor-core convolutions, the reference's own GPU arithmetic (torch cudnn.allow_tf32 "
                          "default); bf16 legs are reported under `legs` and are backed by tests/test_gpu_attack_success.py",
    }

    def k1_leg_roofline(eng, wl):
        """K1 (expand_kernel<FUSED=1>) on the launch shape this workload's step uses: CUDA events around 10 back-to-back launches
        rotating over > 400 MB of outputs, median of 5; algorithmic bytes = 3*H*W*elem per sample + 7 fp32 planes per image."""
        import ctypes as C
        from dorpatch_b200 import _lib
        B, S_loc, es = wl.B, wl.S_loc, eng.elem_bytes
        n = int(eng.lib.dp_k1_samples_per_launch(eng.handle, B * S_loc))
        rects = wl.PM.gather(wl.table, np.stack([np.random.RandomState(b).choice(wl.n_mask, S_loc, replace=False) for b in range(B)]))
        rd = torch.from_numpy(np.ascontiguousarray(rects.reshape(B * S_loc, 4, 4), np.int16)).to(dev)
        dt_t = torch.bfloat16 if es == 2 else torch.float32
        n_rot = max(2, int(400e6 // (n * IMG * IMG * eng.c_pad * es)) + 1)
        bufs = [torch.empty((n, IMG, IMG, eng.c_pad), dtype=dt_t, device=dev) for _ in range(n_rot)]
        eng.paste(wl.x, wl.mask, wl.pattern, 4.0)
        starts = list(range(0, B * S_loc - n + 1, n)) or [0]
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def launch(i):
            _lib.check(eng.lib.dp_expand_step_dev(eng.handle, C.c_void_p(wl.x.data_ptr()), C.c_void_p(wl.mask.data_ptr()), C.c_void_p(wl.pattern.data_ptr()),
                                                  B, S_loc, C.c_void_p(rd.data_ptr()), starts[i % len(starts)], n, C.c_void_p(bufs[i % n_rot].data_ptr()), eng._stream()))
        for i in range(4):
            launch(i)
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            ev0.record()
            for i in range(10):
                launch(i)
            ev1.record()
            torch.cuda.synchronize()
            ts.append(ev0.elapsed_time(ev1) / 10)
        ms = float(np.median(ts))
        alg = n * IMG * IMG * 3 * es + max(1, n // S_loc) * 7 * IMG * IMG * 4
        phys = n * IMG * IMG * eng.c_pad * es + max(1, n // S_loc) * 7 * IMG * IMG * 4
        del bufs
        return {"frac": alg / ms / 1e6 / pk["hbm"], "frac_physical": phys / ms / 1e6 / pk["hbm"], "achieved_gbs": alg / ms / 1e6, "ms": ms, "samples_per_launch": n, "c_pad": eng.c_pad}

    def kernel_table(eng, wl, i):
        eng.profile(True, reset=True)
        wl.step(i)
        torch.cuda.synchronize()
        prof = eng.profile_read()
        eng.profile(False)
        tot = sum(v["ms"] for v in prof.values()) or 1.0
        kern = {}
        for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
            d = {"ms": round(v["ms"], 3), "share": round(v["ms"] / tot, 4), "launch_groups": v["count"]}
            if v["flops"] > 0 and ("conv" in k or "gemm" in k):
                d["tflops"] = round(v["flops"] / v["ms"] / 1e9, 1)
                d["frac_of_bf16_peak"] = round(v["flops"] / v["ms"] / 1e9 / pk["tf_burst"], 3)
                if v["bytes"] > 0:        # these layers are HBM-bound in this network (33 FLOP/B): the byte rate is the telling one
                    d["gbs_algorithmic"] = round(v["bytes"] / v["ms"] / 1e6, 1)
                    d["frac_of_hbm_peak"] = round(v["bytes"] / v["ms"] / 1e6 / pk["hbm"], 3)
            else:
                d["gbs_algorithmic"] = round(v["bytes"] / v["ms"] / 1e6, 1)
                d["frac_of_hbm_peak"] = round(v["bytes"] / v["ms"] / 1e6 / pk["hbm"], 3)
            kern[k] = d
        return kern, round(tot, 3)

    # profiled step (all ranks execute it to keep collectives matched)
    kern, ktot = kernel_table(eng, wl, W + 2 * K + 10)

    if rank == 0:
        es = eng.elem_bytes
        # ---- K1 roofline: the variant the step launches (paste fused in, 7 input planes, one launch per classifier chunk)
        #      on exactly that launch shape; CUDA events around back-to-back launches over rotating outputs > L2 --------
        import ctypes as C
        from dorpatch_b200 import _lib
        B, S_loc = wl.B, wl.S_loc
        n_chunk = int(eng.lib.dp_k1_samples_per_launch(eng.handle, B * S_loc))       # what ONE K1 launch of the step covers
        rects_all = wl.PM.gather(wl.table, np.stack([np.random.RandomState(b).choice(wl.n_mask, S_loc, replace=False) for b in range(B)]))
        ra_dev = torch.from_numpy(np.ascontiguousarray(rects_all.reshape(B * S_loc, 4, 4), np.int16)).to(dev)
        dt_t = torch.bfloat16 if es == 2 else torch.float32
        n_rot = max(2, int(400e6 // (n_chunk * IMG * IMG * eng.c_pad * es)) + 1)      # rotate over > 400 MB of outputs (> L2)
        bufs = [torch.empty((n_chunk, IMG, IMG, eng.c_pad), dtype=dt_t, device=dev) for _ in range(n_rot)]
        eng.paste(wl.x, wl.mask, wl.pattern, 4.0)                                 # the clip scale the fused variant reads
        n_starts = list(range(0, B * S_loc - n_chunk + 1, n_chunk)) or [0]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def k1_launch(i, rp):
            _lib.check(eng.lib.dp_expand_step_dev(eng.handle, C.c_void_p(wl.x.data_ptr()), C.c_void_p(wl.mask.data_ptr()),
                                                  C.c_void_p(wl.pattern.data_ptr()), B, S_loc, rp, n_starts[i % len(n_starts)], n_chunk,
                                                  C.c_void_p(bufs[i % n_rot].data_ptr()), eng._stream()))

        def k1_time(rp, pairs, per_pair=10):
            for i in range(4):
                k1_launch(i, rp)
            torch.cuda.synchronize()
            ts = []
            for _ in range(pairs):
                e0.record()
                for i in range(per_pair):
                    k1_launch(i, rp)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1) / per_pair)
            return float(np.median(ts))

        rp_dev = C.c_void_p(ra_dev.data_ptr())
        k1_ms = k1_time(rp_dev, 7)
        k1_ms_clean = k1_time(None, 3)                         # diagnostic: same launch without occluders (pure bulk-store path)
        e0.record(); k1_launch(0, rp_dev); e1.record(); torch.cuda.synchronize()
        k1_ms_single = e0.elapsed_time(e1)
        img_in_launch = max(1, n_chunk // S_loc)
        alg_bytes = n_chunk * IMG * IMG * 3 * es + img_in_launch * 7 * IMG * IMG * 4
        traffic, tnote = None, None
        tpath = os.path.join(ROOT, "profiles", "k1_traffic.json")     # dram bytes of this launch from the last ncu --set full capture
        if os.path.exists(tpath):
            for tj in json.load(open(tpath)).get("entries", []):
                if tj.get("samples") == n_chunk and tj.get("dtype") == args.precision:
                    traffic, tnote = tj.get("dram_bytes"), tj.get("note")
        phys_bytes = n_chunk * IMG * IMG * eng.c_pad * es + img_in_launch * 7 * IMG * IMG * 4
        out["roofline"] = {"kernel": "expand_kernel<FUSED=1> (K1: paste + L2-scale + normalise + occlude, TMA bulk tiles), the in-step variant and launch shape (%d samples per launch)" % n_chunk,
                           "physical_bytes_per_launch": phys_bytes, "frac_physical": phys_bytes / k1_ms / 1e6 / pk["hbm"],
                           "physical_note": "bytes the launch really moves: the network input is [N,H,W,%d] (channel pad %d -> %d for the library stem)" % (eng.c_pad, 3, eng.c_pad) if eng.c_pad != 3 else "tight C=3 layout: physical == algorithmic",
                           "bound": "hbm", "achieved": alg_bytes / k1_ms / 1e6, "peak": pk["hbm"], "unit": "GB/s",
                           "frac": alg_bytes / k1_ms / 1e6 / pk["hbm"], "traffic": traffic, "traffic_note": tnote,
                           "ms": k1_ms, "ms_single_launch_event_pair": k1_ms_single, "samples_per_launch": n_chunk,
                           "timing": "CUDA events around 10 back-to-back launches rotating over %d output buffers (> L2 in total), median of 7" % n_rot,
                           "unoccluded_gbs": alg_bytes / k1_ms_clean / 1e6,
                           "algorithmic_bytes_per_launch": alg_bytes,
                           "algorithmic_bytes_per_unit": "3*224*224*%d B written per EOT sample + 7*224*224*4 B read per image (SURVEY 8d)" % es,
                           "peak_source": pk["src"]}
        del bufs
        out["roofline_step"] = {"bound": "tensor", "achieved": GFLOP_PER_SAMPLE * head["value"] / world / 1e3, "peak": pk["tf_sus"],
                                "unit": "TFLOP/s", "frac": GFLOP_PER_SAMPLE * head["value"] / world / 1e3 / pk["tf_sus"],
                                "note": "16.36 GFLOP (fwd+dgrad) per EOT sample x per-GPU samples/s vs sustained bf16 cuBLAS peak (TF32 peak is half of it)"}
        out["kernels"] = kern
        out["kernels_total_ms"] = ktot
        out["kernels_note"] = "one step profiled with CUDA events around every launch, chunks serialised on ONE lane; the timed steps overlap two lanes (two streams), so ms_per_step < kernels_total_ms"
        # ---- forward-only universe scan (collect_failure, attack.py:384-406) + PatchCleanser evaluation (c3 names it) ----
        try:
            Bs = 4
            rects_scan = wl.PM.gather(wl.table, np.tile(np.arange(wl.n_mask), (Bs, 1)))
            eng.predict(wl.x[:Bs], wl.n_mask, rects_scan)
            ts = []
            for _ in range(3):
                e0.record(); eng.predict(wl.x[:Bs], wl.n_mask, rects_scan); e1.record(); torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            scan_ms_img = float(np.median(ts)) / Bs
            amort = wl.samples_per_step / ((head["ms_per_step"] + scan_ms_img * wl.B / 100.0 / world) / 1e3)
            out["scan"] = {"fwd_samples_per_s": wl.n_mask / (scan_ms_img / 1e3), "masks": int(wl.n_mask), "ms_per_image": scan_ms_img,
                           "amortised_eot_samples_per_s": amort,
                           "note": "dp_predict over the whole mask universe; amortised = `value` with one scan per image every 100 steps added (attack.py:187-190), the universe split over the ranks"}
            out["value_scan_amortised"] = amort
            from dorpatch_b200.defenses.PatchCleanser import MaskWindow, PatchCleanser
            from dorpatch_b200.utils import NormModel, get_normalize
            import contextlib, io
            net_native = ResNetV2(seed=0)
            net_native._engines = {}
            model = torch.nn.DataParallel(NormModel(net_native, get_normalize("imagenet", "resnetv2")))
            net_native.adopt_engine(eng)
            with contextlib.redirect_stdout(io.StringIO()):
                defs = [PatchCleanser(MaskWindow(IMG, r, 1), model) for r in (0.015, 0.03, 0.06, 0.12)]
            l0 = eng.launch_count
            t0 = time.perf_counter()
            n_img = 2
            for im in wl.x[:n_img]:
                for d in defs:
                    d.robust_predict(im, True)
            torch.cuda.synchronize()
            dtp = time.perf_counter() - t0
            out["patchcleanser_eval"] = {"images_per_s": n_img / dtp, "ms_per_image_4_ratios": dtp / n_img * 1e3,
                                         "note": "defenses/PatchCleanser.py:68-112 on dp_predict: 36 single + 630 double masks (+ second round) x 4 ratios per image (main.py:61,151)"}
        except Exception as ex:                                             # side figures: never lose the bench line over them
            out.setdefault("scan", {"error": str(ex)[:300]})
            out["patchcleanser_eval"] = {"error": str(ex)[:300]}
    del wl
    # ---- extra legs (single GPU only; each is a full timed run of K steps) -----------------------------------------------
    if world == 1 and not args.no_legs:
        legs = {}
        other = "bf16" if args.precision != "bf16" else "tf32"
        plan = [(args.precision, "c2"), (args.precision, "b1"), (args.precision, "c5s0"), (other, "c3"), (other, "c2"), (other, "b1")]
        for prec, cfg in plan:
            if cfg == args.config and prec == args.precision:
                continue
            try:
                r = measure(prec, cfg, K, e2e=(cfg in ("c2", "c3")))
                leg = {"value": r["value"], "ms_per_step": r["ms_per_step"], "gpu_launches": r["launches"], "dtype": prec, "host_ms_per_step": r["host_ms"],
                       "config": workload_config(cfg, 1)["workload"]}
                if "e2e_value" in r:
                    leg["e2e"] = r["e2e_value"]
                if cfg == "c2" and prec == "bf16":
                    leg["kernels"], leg["kernels_total_ms"] = kernel_table(r["eng"], r["wl"], 900)   # i < 1000: no failed-set sampling (as every timed step)
                legs["%s_%s" % (prec, cfg)] = leg
                if cfg in ("c3", "c2"):          # K1 roofline of this leg's in-step launch (same method as the headline `roofline`)
                    try:
                        leg["k1_roofline"] = k1_leg_roofline(r["eng"], r["wl"])
                    except Exception as ex:
                        leg["k1_roofline"] = {"error": str(ex)[:200]}
                del r
            except Exception as ex:
                legs["%s_%s" % (prec, cfg)] = {"error": str(ex)[:300]}
        out["legs"] = legs
    for e in engines.values():
        e.close()
    if rank == 0:
        # ---- CPU baseline: oracle port on this box's host cores, bounded sample ----------------------------
        if world == 1 and not args.no_cpu_baseline:
            try:
                S = CONFIGS[args.config]["S"]
                cstep, threads = cpu_step_factory(S)
                cstep()
                t0, n = time.perf_counter(), 0
                while time.perf_counter() - t0 < args.cpu_seconds:
                    n += cstep()
                dtc = time.perf_counter() - t0
                out["cpu_baseline"] = {"value": n / dtc, "unit": UNIT, "cores": threads, "kind": "port",
                                       "sample": "%d steps of 1 image x %d EOT samples (%.1f s), stage-1 step, fp32 torch-CPU oracle port, weight grads on as in the reference" % (n // S, S, dtc)}
            except Exception as ex:   # the bench line must survive a CPU-side problem
                out["cpu_baseline"] = {"error": repr(ex)}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--precision", default=os.environ.get("DORPATCH_BENCH_PRECISION", "tf32"), choices=["fp32", "tf32", "bf16"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--chunk", type=int, default=int(os.environ.get("DORPATCH_CHUNK", "256")))
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-legs", action="store_true", help="skip the extra legs (bf16 / c2 / B=1 / stage 0)")
    ap.add_argument("--ncu", action="store_true", help="run W warm-up steps, then ONE step inside cudaProfilerStart/Stop, and exit")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "native" or args.ncu):
        ap.error("--dump-outputs dumps the native arm's timed steps: it needs --impl native and no --ncu")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
