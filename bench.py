#!/usr/bin/env python
"""bench.py — causal-OT loss forward+backward evaluations per second (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one eval = `compute_sinkhorn_loss` value + gradients w.r.t. f_fake, h_fake, m_real,
h_real, m_fake (BASELINE.md) on synthetic inputs.  The HEADLINE line is BASELINE config 2 (GQN Mazes:
B=64, 3+7 frames of 64x64x3, J=8); with N GPUs every rank evaluates its own independent batch
(problem-parallel, no data-path collective: SURVEY.md §8e) -> weak scaling, value = N*K / max-over-ranks time.

Prints ONE JSON line (rank 0):
  value        inputs resident in HBM, CUDA events, inputs rotated over more data than L2 holds
  e2e          the same call with HOST (pinned) inputs, H2D copies and the D2H read of the loss inside the timed region
  roofline     the dominant HBM-bound kernel of the headline config
  cpu_baseline the reference formulation (oracle/port_torch.py) on the box's host cores
  configs      every other BASELINE config on the same box (value, parity, roofline):
                 cfg1_mmnist  replicas (weak), loss only
                 cfg3_bair    replicas (weak), temporal kernel smoothing of real and fake (fwd + bwd) inside the step
                 cfg4_batched 256 independent problems split over the N ranks (strong), batched C-ABI call
                 cfg5_large   ONE B=8192 problem; N=1: whole problem on the GPU; N>1: cost rows sharded over the
                              ranks, column sums exchanged inside the persistent Sinkhorn kernel (strong)
  notes        how the numbers were taken (L2 policy, launch mode, parallelism)
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

S = 1.0 / 15.0
METRIC = "causal_ot_loss_fwd_bwd_evals_per_sec"
UNIT = "evals/s"
NLANES = 8          # independent evaluations in flight (kccotgan_b200.graphed.EvaluationLanes)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2_mazes")
    ap.add_argument("--kind", default="uniform", choices=["uniform", "video"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager", action="store_true", help="time eager Python calls instead of CUDA-graph replays")
    ap.add_argument("--cpu-budget-s", type=float, default=25.0)
    ap.add_argument("--configs", default="cfg1_mmnist,cfg2_shared_ctx,cfg3_bair,cfg4_batched,cfg5_large",
                    help="comma list of the other BASELINE configs carried in the line ('' = headline only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and gradients of the last timed headline step as DIR/<name>.npy (rank 0)")
    return ap.parse_args()


def workload_config(name, kind):
    from kccotgan_b200.synthetic import CONFIGS
    c = dict(CONFIGS[name])
    nprob = c.pop("nprob", None)
    K = c["T"] * c["H"] * c["W"] * c["C"]
    tag = f"{nprob} x " if nprob else ""
    return c, K, {"workload": f"{name}: {tag}B={c['B']} T={c['T']} ({c['ctx']}+{c['T'] - c['ctx']}) frames "
                              f"{c['H']}x{c['W']}x{c['C']} J=8 s=1/15 eps=1.0 L=100 ({kind} inputs)",
                  "B": c["B"], "K": K, "T": c["T"], "J": 8, "inputs": kind}


# ------------------------------------------------------------------------------------------------
# CPU legs (the only places bench.py executes oracle/)
# ------------------------------------------------------------------------------------------------
def cpu_reference_timing(cfg, kind, steps, warmup, budget_s):
    """Times the reference formulation (oracle/port_torch.py: [B,B,T,D] broadcast cost, eager
    logsumexp loop, autograd through the unrolled iterations) in fp32 on all host cores."""
    import torch
    from kccotgan_b200.synthetic import make_inputs
    from oracle import port_torch as pt
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    inp = make_inputs(J=8, kind=kind, seed=1, **cfg)
    args = (inp["real"], inp["fake"], S, inp["h_fake"], inp["m_real"], inp["h_real"], inp["m_fake"])
    t_start = time.perf_counter()
    for _ in range(max(0, min(warmup, 1))):
        pt.mixed_loss_fwd_bwd(*args)
    done, elapsed = 0, 0.0
    while done < max(1, steps):
        t0 = time.perf_counter()
        pt.mixed_loss_fwd_bwd(*args)
        elapsed += time.perf_counter() - t0
        done += 1
        if time.perf_counter() - t_start > budget_s:
            break
    model = "unknown"
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    return {"value": done / elapsed, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{done} full evals of the workload (1 warm-up), fp32, torch-CPU {cores} threads on '{model}'; "
                      "reference formulation restated in oracle/port_torch.py (TensorFlow and /root/reference are "
                      "absent on the GPU box)",
            "s_per_eval": elapsed / done}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg, K, config = workload_config(args.workload, args.kind)
    r = cpu_reference_timing(cfg, args.kind, args.steps, args.warmup, budget_s=150.0)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["s_per_eval"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config, "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        """Clock summary of the samples taken in [t0, t1] (the sampler keeps running)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [l for t, l in list(self.lines) if t0 - 0.05 <= t <= t1 + 0.15] or [l for _, l in list(self.lines)[-3:]]
        for l in rows:
            parts = [p.strip() for p in l.split(",")]
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()


class Ctx:
    """What every leg of the GPU arm needs."""
    pass


_T0 = time.perf_counter()


def progress(msg):
    """Progress on stderr (the JSON line is the only thing on stdout)."""
    if int(os.environ.get("RANK", "0")) == 0:
        sys.stderr.write(f"[bench +{time.perf_counter() - _T0:6.1f}s] {msg}\n")
        sys.stderr.flush()


def barrier(cx):
    cx.torch.cuda.synchronize()
    if cx.world > 1:
        cx.dist.barrier()
        cx.torch.cuda.synchronize()


def max_over_ranks(cx, ms):
    if cx.world > 1:
        t = cx.torch.tensor([ms], device=cx.dev)
        cx.dist.all_reduce(t, op=cx.dist.ReduceOp.MAX)
        ms = float(t)
    return ms


def timed(cx, fn, steps, warmup=3):
    """W untimed + K timed calls of fn(i), bracketed by barriers, CUDA events, max over ranks -> (ms total, clocks)."""
    torch = cx.torch
    for i in range(warmup):
        fn(i)
        if os.environ.get("KCCOT_BENCH_SYNC"):              # debugging aid: find the call that does not come back
            torch.cuda.synchronize()
            progress(f"warm-up call {i} done")
    barrier(cx)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(steps):
        fn(warmup + i)
    e1.record()
    barrier(cx)
    t1 = time.perf_counter()
    ms = max_over_ranks(cx, e0.elapsed_time(e1))
    return ms, (cx.sampler.window(t0, t1) if cx.rank == 0 else None)


def capture(cx, fn):
    """CUDA graph of fn() (a Python closure over static tensors); returns (replay, outputs) or (None, None)."""
    torch = cx.torch
    try:
        side = torch.cuda.Stream(device=cx.dev)
        side.wait_stream(torch.cuda.current_stream(cx.dev))
        with torch.cuda.stream(side):
            for _ in range(2):
                fn()
        torch.cuda.current_stream(cx.dev).wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = fn()
        return g.replay, out
    except Exception as e:                                   # capture is an optimisation of the launch path only
        sys.stderr.write(f"[bench] graph capture failed ({type(e).__name__}: {e}); timing eager calls\n")
        torch.cuda.synchronize()
        return None, None


def golden_terms(name):
    import numpy as np
    path = os.path.join(ROOT, "tests", "golden", name)
    if not os.path.isfile(path):
        return None
    with np.load(path, allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE = 1 << 20          # elements kept of each large output when the whole set would exceed the limit
GRAD_OUTPUTS = ("fake", "h_fake", "m_real", "h_real", "m_fake")     # the leaves the headline step differentiates


def host_outputs(loss, grads):
    """The arrays a caller of the headline step receives: the loss and the gradients w.r.t. GRAD_OUTPUTS (in that
    order), copied to host memory in their compute dtype (float32)."""
    out = {"loss": loss.detach().cpu().numpy()}
    out.update({"grad_" + n: g.detach().cpu().numpy() for n, g in zip(GRAD_OUTPUTS, grads)})
    return out


def dump_outputs(path, arrays):
    """DIR/<name>.npy for every array.  If the set exceeds DUMP_LIMIT_BYTES, each array larger than DUMP_SAMPLE
    elements is replaced by the same seeded sample of its flattened elements on every run (indices ascending)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    sample = sum(a.nbytes for a in arrays.values()) > DUMP_LIMIT_BYTES
    for name, a in arrays.items():
        if sample and a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a)


def peaks():
    p = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
    except OSError:
        pass
    return p


# ------------------------------------------------------------------------------------------------
# the other BASELINE configs
# ------------------------------------------------------------------------------------------------
def loss_parity(cx, name, kind, prefix=""):
    """Loss terms on the golden's seeded inputs against the committed output of the reference's own source
    (tests/golden, generator oracle/make_golden.py); the full gradient checks live in tests/."""
    from kccotgan_b200 import gan_utils
    from kccotgan_b200.synthetic import CONFIGS, INPUT_ORDER, make_inputs
    g = golden_terms(f"loss_{name}_full_{kind}.npz")
    if g is None:
        return {"checked": False, "why": "no golden fixture for this config / input kind"}
    c = {k: v for k, v in CONFIGS[name].items() if k != "nprob"}
    inp = make_inputs(J=8, kind=kind, seed=1, device=cx.dev, **c)
    lv = [inp[k] for k in INPUT_ORDER]
    if prefix:
        from kccotgan_b200.data_utils import KernelSmoothing
        ks = KernelSmoothing(temporal_kernel_size=6, spatial_kernel_size=6)
        lv[0], lv[1] = ks.temporal_convolution(lv[0], 5.0), ks.temporal_convolution(lv[1], 5.0)
    loss, terms = gan_utils.sinkhorn_loss_terms(lv[0], lv[1], S, *lv[2:])
    ref = [float(g[prefix + "loss_xy"]), float(g[prefix + "loss_xx"]), float(g[prefix + "loss_yy"])]
    scale = max(abs(v) for v in ref)
    err = max(abs(float(a) - b) for a, b in zip(terms.tolist(), ref)) / scale
    lerr = abs(float(loss) - float(g[prefix + "loss"])) / scale
    return {"checked": True, "ok": bool(err <= 1e-4 and lerr <= 1e-4), "max_term_rel_err": err, "loss_rel_err": lerr,
            "against": f"tests/golden/loss_{name}_full_{kind}.npz ({prefix or 'loss'} of the reference's own source, fp64)"}


def run_replica_config(cx, name, kind, steps, smooth):
    """cfg1 / cfg3: independent batch per rank, graph replay of the whole step."""
    torch = cx.torch
    from kccotgan_b200 import gan_utils
    from kccotgan_b200.data_utils import KernelSmoothing
    from kccotgan_b200.synthetic import INPUT_ORDER, make_inputs
    cfg, K, config = workload_config(name, kind)
    B, T = cfg["B"], cfg["T"]
    in_bytes = 2 * B * K * 4
    nsets = max(NLANES, int(300e6 // in_bytes) + 1)
    ks = KernelSmoothing(temporal_kernel_size=6, spatial_kernel_size=6)       # kernel_train.py:216
    steps_fns = []
    for i in range(nsets):
        inp = make_inputs(J=8, kind=kind, seed=1 + cx.rank + 1000 * i, device=cx.dev, **cfg)
        lv = [inp[k].requires_grad_(k != "real") for k in INPUT_ORDER]

        def step(lv=lv):
            real, fake = lv[0], lv[1]
            if smooth:                                      # kernel_train.py:270-279 with --kernel 1d, sigma = 5
                real, fake = ks.temporal_convolution(real, 5.0), ks.temporal_convolution(fake, 5.0)
            loss = gan_utils.compute_sinkhorn_loss(real, fake, S, 0.8, 100, *lv[2:], video=True)
            return loss, torch.autograd.grad(loss, lv[1:])
        steps_fns.append(step)
    replays = []
    for fn in steps_fns:
        r, _ = capture(cx, fn)
        replays.append(r)
    use_graph = all(r is not None for r in replays)
    launches0 = cx.lib.kccot_launch_count()
    steps_fns[0]()
    per_step = int(cx.lib.kccot_launch_count() - launches0)
    serial = None
    if use_graph:
        # independent evaluations replayed round-robin on NLANES streams (see the headline); serial replays beside it
        nl = min(NLANES, nsets)
        streams = [torch.cuda.Stream(cx.dev) for _ in range(nl)]

        def run_lanes(i):
            j = i % nsets
            with torch.cuda.stream(streams[j % nl]):
                replays[j]()

        def timed_lanes(n):
            barrier(cx)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            main = torch.cuda.current_stream(cx.dev)
            t0 = time.perf_counter()
            e0.record(main)
            for s_ in streams:
                s_.wait_stream(main)
            for i in range(n):
                run_lanes(i)
            for s_ in streams:
                main.wait_stream(s_)
            e1.record(main)
            barrier(cx)
            t1 = time.perf_counter()
            return max_over_ranks(cx, e0.elapsed_time(e1)), (cx.sampler.window(t0, t1) if cx.rank == 0 else None)

        timed_lanes(3)
        ms, clocks = timed_lanes(steps)
        ms_s, _ = timed(cx, lambda i: replays[i % nsets](), min(steps, 100))
        serial = cx.world * min(steps, 100) / (ms_s * 1e-3)
    else:
        ms, clocks = timed(cx, lambda i: steps_fns[i % nsets](), steps)
    value = cx.world * steps / (ms * 1e-3)
    alg = 20.0 * B * K + 40.0 * B * T * 8 + (24.0 * B * K if smooth else 0.0)    # SURVEY §8d; 1d smoothing: 3 x 8BK
    hbm = float(peaks().get("hbm_gbs", 6650.0))
    ach = alg / (ms * 1e-3 / steps) / 1e9
    out = {"value": value, "unit": UNIT, "steps": steps, "ms_per_step": ms / steps, "scaling": "weak",
           "config": config, "clocks": clocks, "gpu_launches_per_step": per_step,
           "launch": (f"CUDA-graph replay, {min(NLANES, nsets)} independent evaluations in flight on as many streams"
                      if use_graph else "eager Python calls"),
           "serial_evals_per_s": serial,
           "step": ("temporal_convolution(real), temporal_convolution(fake) -> compute_sinkhorn_loss -> gradients "
                    "to fake (through the smoothing), h_fake, m_real, h_real, m_fake" if smooth else
                    "compute_sinkhorn_loss -> gradients to fake, h_fake, m_real, h_real, m_fake"),
           "roofline": {"bound": "hbm", "scope": "whole step", "achieved": ach, "peak": hbm, "unit": "GB/s",
                        "frac": ach / hbm, "algorithmic_bytes_per_step": alg, "traffic": None}}
    if cx.rank == 0:
        out["parity"] = loss_parity(cx, name, kind, "smooth1d_" if smooth else "")
    return out


def run_shared_ctx(cx, name, steps):
    """SURVEY §8 f3: the same config on video-like inputs (fake shares its context frames with real, as
    kernel_train.py:225-226 builds them), plain call against compute_sinkhorn_loss_shared_context."""
    torch = cx.torch
    from kccotgan_b200.graphed import EvaluationLanes, GraphedSinkhornLoss
    from kccotgan_b200.synthetic import INPUT_ORDER, make_inputs
    cfg, K, config = workload_config(name, "video")
    B, T, ctx = cfg["B"], cfg["T"], cfg["ctx"]
    nsets = NLANES
    out = {"config": config, "ctx_frames": ctx, "unit": UNIT, "steps": steps,
           "launch": f"CUDA-graph replay, {NLANES} independent evaluations in flight"}
    ref = None
    for tag, cf in (("plain", 0), ("shared_context", ctx)):
        evs = []
        for i in range(nsets):
            inp = make_inputs(J=8, kind="video", seed=1 + cx.rank + 1000 * i, device=cx.dev, **cfg)
            evs.append(GraphedSinkhornLoss(*[inp[k] for k in INPUT_ORDER], S, adopt=True, ctx_frames=cf))
        lanes = EvaluationLanes(evs, NLANES)

        def run(n):
            barrier(cx)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            lanes.fork()
            for i in range(n):
                lanes.submit(i % nsets)
            lanes.join()
            e1.record()
            barrier(cx)
            return max_over_ranks(cx, e0.elapsed_time(e1))
        run(6)
        ms = run(steps)
        out[tag] = {"value": cx.world * steps / (ms * 1e-3), "ms_per_step": ms / steps}
        if ref is None:
            ref = (float(evs[0].loss), evs[0].grads["fake"][:, :, ctx:].clone())
        else:
            out["parity"] = {"checked": True,
                             "ok": bool(float(evs[0].loss) == ref[0] and torch.equal(evs[0].grads["fake"][:, :, ctx:], ref[1])),
                             "against": "the plain call on the same inputs: loss and gradient of the predicted frames "
                                        "bit-identical (tests/test_gpu_parity.py::test_shared_context_hint)"}
        del evs, lanes
        torch.cuda.empty_cache()
    out["value"] = out["shared_context"]["value"]
    alg_plain = 20.0 * B * K
    alg_ctx = B * K * (4.0 + 4.0 * (T - ctx) / T + 12.0 * (T - ctx) / T)
    out["algorithmic_bytes_per_step"] = {"plain": alg_plain, "shared_context": alg_ctx}
    hbm = float(peaks().get("hbm_gbs", 6650.0))
    ach = alg_ctx / (out["shared_context"]["ms_per_step"] * 1e-3) / 1e9
    out["roofline"] = {"bound": "hbm", "scope": "whole step", "achieved": ach, "peak": hbm, "unit": "GB/s",
                       "frac": ach / hbm, "traffic": None}
    return out


def run_cfg4(cx, kind, steps):
    """256 independent problems, dealt to the ranks (no collective), one batched C-ABI call per direction."""
    torch = cx.torch
    from kccotgan_b200 import functional as F, gan_utils
    from kccotgan_b200.synthetic import CONFIGS, make_inputs
    cfg, K, config = workload_config("cfg4_batched", kind)
    nprob_total = CONFIGS["cfg4_batched"]["nprob"]
    B, T = cfg["B"], cfg["T"]
    mine = list(range(cx.rank, nprob_total, cx.world))
    P = len(mine)
    nsets = 3
    sets = []
    for s_i in range(nsets):
        g = torch.Generator(device=cx.dev).manual_seed(17 + 1000 * s_i + cx.rank)
        real = torch.rand((P, B, cfg["H"], T, cfg["W"], cfg["C"]), generator=g, device=cx.dev)
        fake = torch.rand((P, B, cfg["H"], T, cfg["W"], cfg["C"]), generator=g, device=cx.dev).requires_grad_(True)
        hm = [torch.sigmoid(torch.randn((P, B, T, 8), generator=g, device=cx.dev)).requires_grad_(True) for _ in range(4)]
        sets.append((real, fake, *hm))
    ones = torch.ones(P, device=cx.dev)

    def make_step(t):
        def step():
            loss = gan_utils.compute_sinkhorn_loss_batched(t[0], t[1], S, *t[2:])
            return loss, torch.autograd.grad(loss, t[1:], grad_outputs=ones)
        return step
    fns = [make_step(t) for t in sets]
    progress(f"cfg4: {P} problems on this rank, {nsets} input sets; capturing")
    replays = [capture(cx, fn)[0] for fn in fns]
    progress("cfg4: captured")
    use_graph = all(r is not None for r in replays)
    n0 = cx.lib.kccot_launch_count()
    loss0, _ = fns[0]()
    per_step = int(cx.lib.kccot_launch_count() - n0)
    if os.environ.get("KCCOT_BENCH_SYNC"):
        torch.cuda.synchronize()
        progress("cfg4: eager call done")
    serial = None
    if use_graph:
        # consecutive steps are independent batches: one stream per input set, so the Sinkhorn kernels of one batch
        # (latency chains, one or two CTAs per SM) run under the HBM kernels of the next
        streams = [torch.cuda.Stream(cx.dev) for _ in range(nsets)]

        def timed_lanes(n):
            barrier(cx)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            main = torch.cuda.current_stream(cx.dev)
            t0 = time.perf_counter()
            e0.record(main)
            for s_ in streams:
                s_.wait_stream(main)
            for i in range(n):
                with torch.cuda.stream(streams[i % nsets]):
                    replays[i % nsets]()
            for s_ in streams:
                main.wait_stream(s_)
            e1.record(main)
            barrier(cx)
            t1 = time.perf_counter()
            return max_over_ranks(cx, e0.elapsed_time(e1)), (cx.sampler.window(t0, t1) if cx.rank == 0 else None)

        timed_lanes(3)
        ms, clocks = timed_lanes(steps)
        ms_s, _ = timed(cx, lambda i: replays[i % nsets](), max(3, min(steps, 20)))
        serial = nprob_total * max(3, min(steps, 20)) / (ms_s * 1e-3)
    else:
        ms, clocks = timed(cx, lambda i: fns[i % nsets](), steps)
    value = nprob_total * steps / (ms * 1e-3)
    alg = (20.0 * B * K + 40.0 * B * T * 8) * P            # per rank and step
    hbm = float(peaks().get("hbm_gbs", 6650.0))
    ach = alg / (ms * 1e-3 / steps) / 1e9
    out = {"value": value, "unit": UNIT + " (problem evaluations)", "steps": steps, "ms_per_step": ms / steps,
           "scaling": "strong", "problems_per_rank": P, "config": config, "clocks": clocks,
           "gpu_launches_per_step": per_step,
           "launch": (f"CUDA-graph replay, {nsets} independent batches in flight on as many streams" if use_graph
                      else "eager Python calls"),
           "serial_evals_per_s": serial,
           "roofline": {"bound": "hbm", "scope": "whole step, per GPU", "achieved": ach, "peak": hbm, "unit": "GB/s",
                        "frac": ach / hbm, "algorithmic_bytes_per_step": alg, "traffic": None}}
    if cx.rank == 0:
        # parity: two of the problems again through the single-problem CUDA-core path (direct (x - y)^2 form)
        F.set_path("simt")
        errs = []
        for q in (0, P - 1):
            t = sets[0]
            l1, _ = gan_utils.sinkhorn_loss_terms(t[0][q].detach(), t[1][q].detach(), S, *[h[q].detach() for h in t[2:]])
            errs.append(abs(float(l1) - float(loss0[q])))
        F.set_path("auto")
        scale = float(loss0.detach().abs().max())
        out["parity"] = {"checked": True, "ok": bool(max(errs) <= 1e-4 * max(scale, 1.0)), "max_abs_err": max(errs),
                         "loss_scale": scale, "against": "the same problems through the CUDA-core direct-form kernels "
                         "(the fp64 oracle checks of this shape are in tests/test_gpu_parity.py)"}
    return out


def tensor_peak_probe(cx):
    """fp16 and tf32 dense matmul rates of this GPU (cuBLAS through torch, best of 5 at 8192^3): the measuring stick
    for the tensor-bound config, beside the driver's bf16 figures."""
    torch = cx.torch
    out = {}
    n = 8192
    for tag, dt in (("fp16", torch.float16), ("tf32", torch.float32)):
        a = torch.randn((n, n), device=cx.dev, dtype=dt)
        b = torch.randn((n, n), device=cx.dev, dtype=dt)
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        best = 1e9
        for i in range(7):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            if i >= 2:
                best = min(best, e0.elapsed_time(e1))
        torch.backends.cuda.matmul.allow_tf32 = old
        out[tag + "_tflops"] = 2.0 * n ** 3 / (best * 1e-3) / 1e12
        del a, b
    return out


def run_cfg5(cx, kind, steps):
    """ONE B = 8192 problem.  N = 1: everything on this GPU.  N > 1: rows sharded (kccotgan_b200.sharded)."""
    torch = cx.torch
    from kccotgan_b200 import _lib, functional as F
    cfg, K, config = workload_config("cfg5_large", kind)
    B, T = cfg["B"], cfg["T"]
    if cx.world > 1:
        from kccotgan_b200 import sharded
        if not hasattr(sharded, "ShardedMixedLoss"):
            return {"unavailable": "row-sharded pipeline not built in this tree"}
        return sharded.bench_cfg5(cx, cfg, K, config, steps, S, timed)
    g = torch.Generator(device=cx.dev).manual_seed(1)
    real = torch.rand((B, K), generator=g, device=cx.dev)
    fake = torch.rand((B, K), generator=g, device=cx.dev)
    hm = [torch.sigmoid(torch.randn((B, T, 8), generator=g, device=cx.dev)) for _ in range(4)]
    L = 100
    lib = cx.lib
    saved = torch.empty(lib.kccot_mixed_loss_saved_bytes(1, B, L), dtype=torch.uint8, device=cx.dev)
    ws = torch.empty(lib.kccot_mixed_loss_workspace_bytes(1, B, K, L), dtype=torch.uint8, device=cx.dev)
    out4 = torch.empty(4, device=cx.dev)
    gl = torch.ones(1, device=cx.dev)
    gf = torch.empty((B, K), device=cx.dev)
    gh = [torch.empty((B, T, 8), device=cx.dev) for _ in range(4)]
    st, p = F._stream(cx.dev), F._ptr
    import ctypes

    def step(_i):
        _lib.call("kccot_mixed_loss_fwd", p(real), p(fake), 1, B, K, p(hm[0]), p(hm[1]), p(hm[2]), p(hm[3]), T, 8, S, 1.0,
                  L, p(saved), ctypes.c_void_p(out4.data_ptr()), ctypes.c_void_p(out4.data_ptr() + 4), p(ws),
                  ws.numel(), 0, st)
        _lib.call("kccot_mixed_loss_bwd", p(gl), p(real), p(fake), 1, B, K, p(hm[0]), p(hm[1]), p(hm[2]), p(hm[3]), T, 8,
                  S, 1.0, L, p(saved), None, p(gf), p(gh[0]), p(gh[1]), p(gh[2]), p(gh[3]), p(ws), ws.numel(), 0, st)
    n0 = lib.kccot_launch_count()
    step(0)
    per_step = int(lib.kccot_launch_count() - n0)
    ms, clocks = timed(cx, step, steps, warmup=1)
    value = steps / (ms * 1e-3)
    pk = peaks()
    probe = tensor_peak_probe(cx)
    peak = float(pk.get("bf16_tflops_sustained", 1400.0))
    flops = 10.0 * B * B * K + 10.0 * B * B * (T - 1) * 8
    ach = flops / (ms * 1e-3 / steps) / 1e12
    executed = 24.0 * B * B * K                            # 3 fp16 products x (4 B^2 K forward with symmetry + 4 B^2 K adjoint)
    out = {"value": value, "unit": UNIT, "steps": steps, "ms_per_step": ms / steps, "scaling": "strong", "config": config,
           "clocks": clocks, "gpu_launches_per_step": per_step, "launch": "C-ABI calls (kccot_mixed_loss_fwd / _bwd)",
           "inputs": "one batch resident in HBM (5.4 GB of videos >> L2)",
           "roofline": {"bound": "tensor", "scope": "whole step (cost GEMMs + Sinkhorn + adjoint)", "achieved": ach,
                        "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                        "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (fp16 runs at the bf16 rate; the step is "
                                       "a 0.2 s loop under the power cap)",
                        "algorithmic_flops_per_step": flops,
                        "executed_mma_tflops": executed / (ms * 1e-3 / steps) / 1e12,
                        "executed_mma_frac": executed / (ms * 1e-3 / steps) / 1e12 / peak,
                        "note": "fp32-grade accuracy needs three fp16 products per term (hi.hi, hi.lo, lo.hi), so the "
                                "tensor pipe executes 2.4x the algorithmic flops (24 B^2 K against 10 B^2 K, the symmetric "
                                "xx / yy blocks computed once); the 3-product-effective peak is peak / 2.4",
                        "effective_peak_3products": peak / 2.4, "frac_of_effective_peak": ach / (peak / 2.4),
                        "measured_here": probe, "traffic": None}}
    # parity: a corner of C_xy against the CUDA-core direct (x - y)^2 kernels; loss terms finite
    n = 256
    C3 = saved[: 3 * B * B * 4].view(torch.float32).view(3, B, B)
    Cc = torch.empty((n, n), device=cx.dev)
    wsc = torch.empty(lib.kccot_cost_workspace_bytes(1, n, n, K), dtype=torch.uint8, device=cx.dev)
    r, f = real[:n].contiguous(), fake[:n].contiguous()
    h0, m1 = hm[0][:n].contiguous(), hm[1][:n].contiguous()
    _lib.call("kccot_cost_fwd", p(r), p(f), 1, n, n, K, p(h0), p(m1), None, None, T, 8, S, p(Cc), p(wsc), wsc.numel(), 1, st)
    err = float((C3[0, :n, :n] - Cc).abs().max() / Cc.abs().max())
    fin = bool(torch.isfinite(out4).all() and torch.isfinite(gf).all())
    out["parity"] = {"checked": True, "ok": bool(err < 2e-6 and fin), "cost_corner_max_rel_err": err, "finite": fin,
                     "loss_terms": out4[1:].tolist(),
                     "against": "256 x 256 corner of C_xy through the CUDA-core direct-form kernels (the reference "
                                "formulation needs a 22 TB temporary at this size; fp64 oracle parity of the same kernels "
                                "at B = 128..1024 is in tests/test_gpu_large.py)"}
    return out


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    import torch
    import torch.distributed as dist
    from kccotgan_b200 import _lib, functional as F, gan_utils
    from kccotgan_b200.synthetic import INPUT_ORDER, make_inputs

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: kccotgan_b200 has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    _lib.check(lib.kccot_device_check())
    cfg, K, config = workload_config(args.workload, args.kind)
    B, T = cfg["B"], cfg["T"]
    notes = {}
    dump = bool(args.dump_outputs) and rank == 0

    cx = Ctx()
    cx.torch, cx.dist, cx.world, cx.rank, cx.dev, cx.lib = torch, dist, world, rank, dev, lib
    cx.sampler = ClockSampler(local)
    if rank == 0:
        cx.sampler.start()
        time.sleep(0.3)

    # ---- inputs: NSETS distinct batches so that consecutive steps never find their videos in L2
    in_bytes = 2 * B * K * 4
    nsets = max(NLANES, int(300e6 // in_bytes) + 1)
    nsets = (nsets + NLANES - 1) // NLANES * NLANES          # a multiple of the lanes: a set always replays on the same lane
    sets = []
    for i in range(nsets):
        inp = make_inputs(J=8, kind=args.kind, seed=1 + rank + 1000 * i, device=dev, **cfg)
        sets.append([inp[k].requires_grad_(k != "real") for k in INPUT_ORDER])
    notes["l2_policy"] = f"inputs rotated over {nsets} distinct batches ({nsets * in_bytes / 1e6:.0f} MB > 126 MB L2)"
    notes["parallelism"] = f"problem-parallel x{world} (independent batch per GPU, no collective)"

    def step(leaves):
        loss = gan_utils.compute_sinkhorn_loss(leaves[0], leaves[1], S, 0.8, 100, *leaves[2:], video=True)
        grads = torch.autograd.grad(loss, leaves[1:])
        return loss, grads

    progress(f"headline {args.workload}: {nsets} input sets ready")
    for i in range(max(3, args.warmup)):
        step(sets[i % nsets])
    barrier(cx)
    # one captured graph per input set (static-buffer contract of kccotgan_b200.graphed)
    from kccotgan_b200.graphed import GraphedSinkhornLoss
    graphs = None
    if not args.eager:
        graphs = [GraphedSinkhornLoss(*[t.detach() for t in sets[i]], S, adopt=True) for i in range(nsets)]
        for i in range(max(3, args.warmup)):
            graphs[i % nsets].step()
        barrier(cx)
        # the replayed graph must reproduce the eager result bit for bit
        l_e, g_e = step(sets[0])
        graphs[0].step()
        torch.cuda.synchronize()
        assert float(l_e) == float(graphs[0].loss), (float(l_e), float(graphs[0].loss))
        assert torch.equal(g_e[0], graphs[0].grads["fake"])
        notes["launch"] = "CUDA-graph replay of the fused forward+backward chain (kccotgan_b200.graphed)"
    else:
        notes["launch"] = "eager Python calls (gan_utils.compute_sinkhorn_loss + torch.autograd.grad)"

    progress("graphs captured; timing the headline")
    launches0 = lib.kccot_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    last_eager = []                                 # (loss, grads) of the last eager step, kept only for the dump

    def timed_serial(n):
        barrier(cx)
        t0 = time.perf_counter()
        e0.record()
        for i in range(n):
            if graphs is not None:
                graphs[i % nsets].step()
            elif dump and i == n - 1:
                last_eager[:] = [step(sets[i % nsets])]
            else:
                step(sets[i % nsets])
        e1.record()
        barrier(cx)
        return max_over_ranks(cx, e0.elapsed_time(e1)), t0, time.perf_counter()

    lanes = None
    if graphs is not None:
        # Consecutive steps are independent evaluations (own batch, own buffers): they are replayed round-robin on
        # NLANES streams, so the Sinkhorn kernels of one evaluation (3 SMs) run under the HBM kernels of the others.
        from kccotgan_b200.graphed import EvaluationLanes
        lanes = EvaluationLanes(graphs, NLANES)              # input set j always replays on stream j % NLANES

        def timed_lanes(n):
            barrier(cx)
            t0 = time.perf_counter()
            e0.record()
            lanes.fork()
            for i in range(n):
                lanes.submit(i % nsets)
            lanes.join()
            e1.record()
            barrier(cx)
            return max_over_ranks(cx, e0.elapsed_time(e1)), t0, time.perf_counter()

        timed_lanes(max(3, args.warmup))
        ms, t0, t1 = timed_lanes(args.steps)
        if dump:                                    # before the serial leg replays the graphs again
            last = graphs[(args.steps - 1) % nsets]
            dumped = host_outputs(last.loss, [last.grads[n] for n in GRAD_OUTPUTS])
        ms_serial, _, _ = timed_serial(min(args.steps, 400))
        serial_evals = world * min(args.steps, 400) / (ms_serial * 1e-3)
        # the overlapped replays must leave the same results as a serial replay
        graphs[0].step()
        torch.cuda.synchronize()
        assert float(l_e) == float(graphs[0].loss) and torch.equal(g_e[0], graphs[0].grads["fake"])
        notes["launch"] += (f"; {NLANES} independent evaluations in flight on {NLANES} streams "
                            "(kccotgan_b200.graphed.EvaluationLanes), results bit-identical to serial replays")
    else:
        ms, t0, t1 = timed_serial(args.steps)
        serial_evals = None
        if dump:
            dumped = host_outputs(*last_eager[0])
    launches = lib.kccot_launch_count() - launches0
    if graphs is not None:
        launches = args.steps * graphs[0].kernels_per_replay      # replays do not pass through the C-ABI counter
    clocks = cx.sampler.window(t0, t1) if rank == 0 else None
    value = world * args.steps / (ms * 1e-3)
    eager_evals = None
    if graphs is not None:                          # also report the eager Python path (the reference-signature call)
        ne = max(200, min(args.steps, 500))
        for i in range(10):
            step(sets[i % nsets])
        barrier(cx)
        e0.record()
        for i in range(ne):
            step(sets[i % nsets])
        e1.record()
        barrier(cx)
        eager_evals = world * ne / (max_over_ranks(cx, e0.elapsed_time(e1)) * 1e-3)

    progress(f"headline {value:.0f} evals/s; eager + e2e legs")
    # ---- e2e: host (pinned) inputs through the public API, H2D + D2H inside the timed region
    host = [[t.detach().cpu().pin_memory() for t in sets[i]] for i in range(min(nsets, 3))]
    h2d = sum(t.numel() * 4 for t in host[0])

    # Double-buffered: the H2D copy of step i+1 runs on a copy stream while step i computes; the loss of
    # step i is copied to pinned host memory asynchronously and read one step later (what a training loop
    # that prefetches its next batch and logs its loss does).  Every step still copies its own inputs.
    copy_s = torch.cuda.Stream(dev)
    main_s = torch.cuda.current_stream(dev)
    dbuf = [[torch.empty(t.shape, dtype=t.dtype, device=dev) for t in host[0]] for _ in range(2)]
    ev_copied = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    ev_loss = [torch.cuda.Event() for _ in range(2)]

    def e2e_run(n):
        loss_pin = torch.empty(n, dtype=torch.float32).pin_memory()
        out = []
        for i in range(n):
            b = i % 2
            with torch.cuda.stream(copy_s):
                if i >= 2:
                    copy_s.wait_event(ev_free[b])          # the compute that read this buffer two steps ago is done
                for d, h in zip(dbuf[b], host[i % len(host)]):
                    d.copy_(h, non_blocking=True)
                ev_copied[b].record(copy_s)
            main_s.wait_event(ev_copied[b])
            leaves = [d.detach().requires_grad_(j != 0) for j, d in enumerate(dbuf[b])]
            loss, grads = step(leaves)
            loss_pin[i].copy_(loss.detach(), non_blocking=True)     # D2H read of the loss
            ev_loss[b].record(main_s)
            ev_free[b].record(main_s)
            if i >= 1:
                ev_loss[(i - 1) % 2].synchronize()
                out.append(float(loss_pin[i - 1]))
        ev_loss[(n - 1) % 2].synchronize()
        out.append(float(loss_pin[n - 1]))
        return out

    e2e_run(4)
    barrier(cx)
    n_e2e = max(5, min(args.steps, 40))
    e0.record()
    e2e_losses = e2e_run(n_e2e)
    e1.record()
    barrier(cx)
    assert all(math.isfinite(v) for v in e2e_losses)
    ms_e2e = max_over_ranks(cx, e0.elapsed_time(e1))
    e2e = {"value": world * n_e2e / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
           "steps": n_e2e, "pipeline": "H2D of step i+1 on a copy stream overlaps the compute of step i (2 device "
                                        "buffers); the 4-byte loss is read back one step late; the 31.5 MB gradient "
                                        "stays on the device (it feeds the generator's backward pass there)"}

    # ---- the other BASELINE configs (all ranks take part: barriers and max-over-ranks inside)
    del graphs, dbuf, host
    sets_keep = sets
    torch.cuda.empty_cache()
    other = {}
    wanted = [c for c in args.configs.split(",") if c]
    few = max(3, min(args.steps, 200))
    import faulthandler
    for name in wanted:
        progress(f"config {name}")
        faulthandler.dump_traceback_later(int(os.environ.get("KCCOT_BENCH_TB", "240")), exit=False)   # a stuck leg leaves its Python stack on stderr
        try:
            if name == "cfg1_mmnist":
                other[name] = run_replica_config(cx, name, args.kind, few, smooth=False)
            elif name == "cfg3_bair":
                other[name] = run_replica_config(cx, name, args.kind, few, smooth=True)
            elif name == "cfg2_shared_ctx":
                other[name] = run_shared_ctx(cx, "cfg2_mazes", few)
            elif name == "cfg4_batched":
                other[name] = run_cfg4(cx, args.kind, max(3, min(args.steps, 20)))
            elif name == "cfg5_large":
                other[name] = run_cfg5(cx, args.kind, max(2, min(args.steps, 5)))
        except Exception as e:                       # a failing side config must not take the headline down
            other[name] = {"error": f"{type(e).__name__}: {e}"}
        faulthandler.cancel_dump_traceback_later()
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    progress("stage times, CPU baseline")
    # ---- per-stage device times + roofline of the dominant HBM kernel (rank 0, after the timed region)
    pk = peaks()
    hbm_peak = float(pk.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in pk else "fallback 6.65 TB/s"
    stages = stage_times(lib, F, torch, sets_keep, B, K, T, dev)
    sk_nits = stages.pop("_sinkhorn_nits", None)
    # algorithmic bytes (SURVEY §8d): forward distances read X,Y once (8BK); adjoint reads X,Y and writes g_fake (12BK)
    alg = {"sqdist_tc_kernel": 8.0 * B * K, "grad_tc_kernel": 12.0 * B * K}
    traffic = {}
    try:        # DRAM bytes per launch from the committed `ncu --set full` capture of the same kernels
        with open(os.path.join(ROOT, "profiles", "r2_dram_traffic.json")) as f:
            traffic = json.load(f)
    except OSError:
        pass
    # the dominant kernel = the one that moves most of the evaluation's bytes (the adjoint GEMM: 12 of the 20 B K bytes);
    # the two HBM kernels take about the same time, the other one is listed in `other_hbm_kernels`
    dom = max(alg, key=lambda k: alg[k])
    dur_us = stages[dom]
    achieved = alg[dom] / (dur_us * 1e-6) / 1e9
    roofline = {"kernel": dom, "dominant_by": "algorithmic bytes per launch (12 B K of the evaluation's 20 B K)",
                "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": traffic.get(dom.split("(")[0]), "peak_source": peak_src,
                "traffic_source": "profiles/r2_dram_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum of one "
                                  "`ncu --set full` capture of the same kernel; not re-measured in this run)",
                "other_hbm_kernels": {k: {"achieved_GBps": alg[k] / (stages[k] * 1e-6) / 1e9,
                                          "frac": alg[k] / (stages[k] * 1e-6) / 1e9 / hbm_peak} for k in alg if k != dom},
                "algorithmic_bytes_per_launch": alg[dom], "avg_launch_us": dur_us,
                "stage_us": stages,
                "whole_eval": {"algorithmic_bytes": 20.0 * B * K + 40.0 * B * T * 8,
                               "frac_of_hbm_roofline": (20.0 * B * K + 40.0 * B * T * 8) / (ms * 1e-3 / args.steps) / 1e9
                               / hbm_peak}}

    if sk_nits:
        # The Sinkhorn pair is not a bandwidth kernel: one CTA per problem, every iteration a dependent chain of two
        # mat-vecs through shared memory.  Its roofline is the bare mat-vec loop of scripts/matvec_probe.py
        # (kccot_debug_matvec_probe, development build): 478 cycles per iteration on two lanes per row (forward), 569 on
        # four (backward).  Cycles here = whole launch (prologue and epilogue included) / iterations of the longest solve.
        mhz = float((clocks or {}).get("sm_mhz") or pk.get("sm_max_mhz") or 1965.0)
        nmax = max(1, max(sk_nits))
        fwd_c = stages["sinkhorn_fwd_small_kernel"] * mhz / nmax
        bwd_c = stages["sinkhorn_bwd_small_kernel"] * mhz / nmax
        roofline["sinkhorn"] = {"bound": "on-chip latency (3 CTAs on 3 of 148 SMs)", "iterations": sk_nits,
                                "fwd_cycles_per_counted_iteration": fwd_c, "bwd_cycles_per_step": bwd_c,
                                "floor_cycles": {"fwd (two lanes per row)": 478, "bwd (four lanes per row)": 569},
                                "frac_bwd": 569.0 / bwd_c,
                                "fwd_note": "the forward stops at its bit-exact fixed point (55-71 executed iterations on "
                                            "these inputs) and fills the history up to the counted 100, so its cycles "
                                            "per COUNTED iteration can undercut the floor of an executed one; the "
                                            "backward executes every counted step",
                                "floor_source": "bare mat-vec pair loop, scripts/matvec_probe.py (round 1, DESIGN.md §5)"}
    cpu = None
    if not args.no_cpu_baseline:
        cpu = cpu_reference_timing(cfg, args.kind, steps=3, warmup=1, budget_s=args.cpu_budget_s)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    cx.sampler.stop()

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 (cost GEMMs 3xTF32 / 3xFP16-split on tcgen05, fp32 accumulate)",
            "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu, "eager_evals_per_s": eager_evals,
            "serial_evals_per_s": serial_evals, "lanes": NLANES if serial_evals is not None else 1, "notes": notes,
            "configs": other}
    if dump:
        dump_outputs(args.dump_outputs, dumped)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def stage_times(lib, F, torch, sets, B, K, T, dev, reps=40):
    """CUDA-event time of each stage of one eval, called through the C ABI, inputs cold in L2."""
    from kccotgan_b200 import _lib
    J = 8
    nsets = len(sets)
    C3 = torch.empty(3, B, B, device=dev)
    Cb = torch.empty_like(C3)
    ws = torch.empty(lib.kccot_mixed_cost_workspace_bytes(1, B, K), dtype=torch.uint8, device=dev)
    ws2 = torch.empty(max(256, lib.kccot_sinkhorn_workspace_bytes(3, B, 100)), dtype=torch.uint8, device=dev)
    ws3 = torch.empty(lib.kccot_mixed_cost_bwd_workspace_bytes(1, B, K), dtype=torch.uint8, device=dev)
    uh = torch.empty(3, 101, B, device=dev)
    vh = torch.empty_like(uh)
    nits = torch.empty(3, dtype=torch.int32, device=dev)
    cost = torch.empty(3, device=dev)
    g3 = torch.tensor([2.0, -1.0, -1.0], device=dev)
    gf = torch.empty(B, K, device=dev)
    gh = [torch.empty(B, T, J, device=dev) for _ in range(4)]
    st = F._stream(dev)
    p = F._ptr

    def views(i):
        r, f, hf, mr, hr, mf = [t.detach() for t in sets[i % nsets]]
        return r.reshape(B, -1), f.reshape(B, -1), hf, mr, hr, mf

    def f_partials(i):
        r, f, hf, mr, hr, mf = views(i)
        _lib.call("kccot_mixed_sqdist_partials", p(r), p(f), 1, B, K, p(ws), ws.numel(), 0, st)

    def f_cost(i):
        r, f, hf, mr, hr, mf = views(i)
        _lib.call("kccot_mixed_cost_fwd", p(r), p(f), 1, B, K, p(hf), p(mr), p(hr), p(mf), T, J, S, p(C3), p(ws),
                  ws.numel(), 0, st)

    def f_skf(i):
        _lib.call("kccot_sinkhorn_fwd", p(C3), 3, B, 1.0, 100, 100, 1e-2, 0, p(uh), p(vh), p(nits), p(cost), p(ws2),
                  ws2.numel(), st)

    def f_skb(i):
        _lib.call("kccot_sinkhorn_bwd", p(C3), 3, B, 1.0, 100, p(uh), p(vh), p(nits), p(g3), p(Cb), p(ws2),
                  ws2.numel(), st)

    def f_grad(i):
        r, f, hf, mr, hr, mf = views(i)
        _lib.call("kccot_mixed_cost_bwd", p(Cb), p(r), p(f), 1, B, K, p(hf), p(mr), p(hr), p(mf), T, J, S, None,
                  p(gf), p(gh[0]), p(gh[1]), p(gh[2]), p(gh[3]), p(ws3), ws3.numel(), 0, st)

    def f_grad_only(i):
        r, f, hf, mr, hr, mf = views(i)
        _lib.call("kccot_mixed_cost_bwd", p(Cb), p(r), p(f), 1, B, K, p(hf), p(mr), p(hr), p(mf), T, J, S, None,
                  p(gf), None, None, None, None, p(ws3), ws3.numel(), 0, st)

    out = {}
    for name, fn in (("sqdist_tc_kernel", f_partials), ("cost_fwd(sqdist+finalize)", f_cost),
                     ("sinkhorn_fwd_small_kernel", f_skf), ("sinkhorn_bwd_small_kernel", f_skb),
                     ("cost_bwd(W+grad+martingale)", f_grad), ("grad_tc_kernel", f_grad_only)):
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        # back-to-back launches (input sets rotate, so the videos are cold in L2): launch latency overlaps
        # execution and the event pair brackets `reps` launches on the launching stream
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            fn(i + 3)
        b.record()
        torch.cuda.synchronize()
        out[name] = a.elapsed_time(b) / reps * 1e3
        if name == "sinkhorn_fwd_small_kernel":
            out["_sinkhorn_nits"] = [int(v) for v in nits.tolist()]      # iterations of the solve that was just timed
    # "grad_tc_kernel" is the whole call: build_w_image_kernel (64 blocks, ~2 us) + the gradient GEMM; the ncu launch
    # list separates them
    return out


if __name__ == "__main__":
    main()
