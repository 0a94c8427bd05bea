"""bf16 videos in the mixed loss: three arms on the same inputs, per config.

    python scripts/bf16_bench.py [--steps N] [--repeats R] [--out DIR] [--no-profile]

Arms (every arm evaluates the loss and the gradients of fake, h_fake, m_real, h_real, m_fake):
    fp32      fp32 videos, the fp32 entry points;
    bf16      bf16 videos, the bf16 entry points (native tcgen05 path at these shapes);
    cast      bf16 videos through the caller-side route: .float() both videos, the fp32 call, gradient .to(bf16).
Configs 1, 2, 2 with shared context frames (ctx_frames = 3) and 4 (256 problems of [64, 32*10*32], eager batched call).
Configs 1 and 2 are CUDA graphs (GraphedSinkhornLoss, or the same capture around the cast route), timed serially on
one stream and as 8 EvaluationLanes.  Eight input sets per arm (more than the 126 MB L2 holds at config 2), the arms
alternate inside every repeat, three repeats; evaluations per second from CUDA events.  A separate pass records
per-kernel device times with torch.profiler (mean microseconds per evaluation).  The card name and power limit are
printed first.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kccotgan_b200 import _lib, gan_utils  # noqa: E402
from kccotgan_b200.graphed import EvaluationLanes, GraphedSinkhornLoss  # noqa: E402
from kccotgan_b200.synthetic import CONFIGS, INPUT_ORDER, make_inputs  # noqa: E402

S = 1.0 / 15.0
NSETS = 8
ARMS = ("fp32", "bf16", "cast")
BF = torch.bfloat16


class CastRoute:
    """The route open to a bf16 caller without bf16 entry points, captured like GraphedSinkhornLoss: widen both videos,
    the fp32 loss and gradients, narrow the video gradient."""

    def __init__(self, inp, ctx_frames):
        self.bufs = [inp[k].detach().clone() for k in INPUT_ORDER]
        self.ctx_frames = ctx_frames
        for t in self.bufs[2:]:
            t.requires_grad_(True)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self._eager()
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss, self.grads = self._eager()

    def _eager(self):
        real, fake = self.bufs[0].float(), self.bufs[1].float().requires_grad_(True)
        hf, mr, hr, mf = self.bufs[2:]
        if self.ctx_frames:
            loss, _ = gan_utils.compute_sinkhorn_loss_shared_context(real, fake, S, hf, mr, hr, mf, self.ctx_frames)
        else:
            loss = gan_utils.compute_sinkhorn_loss(real, fake, S, 0.8, 100, hf, mr, hr, mf)
        g = torch.autograd.grad(loss, [fake, hf, mr, hr, mf])
        return loss, (g[0].to(BF), *g[1:])


def _graph(arm, inp, ctx_frames):
    if arm == "cast":
        return CastRoute(inp, ctx_frames)
    d = {k: v.detach().clone() for k, v in inp.items()}
    if arm == "fp32":
        d["real"], d["fake"] = d["real"].float(), d["fake"].float()
    return GraphedSinkhornLoss(*[d[k] for k in INPUT_ORDER], S, adopt=True, ctx_frames=ctx_frames)


def _time(fn, steps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3


def graph_config(name, ctx_frames, steps, repeats):
    c = {k: v for k, v in CONFIGS[name].items() if k not in ("nprob", "ctx")}
    sets = []
    for i in range(NSETS):
        d = make_inputs(J=8, kind="video" if ctx_frames else "uniform", ctx=ctx_frames or None, seed=1 + 1000 * i,
                        device="cuda", **c)
        d["real"], d["fake"] = d["real"].to(BF), d["fake"].to(BF)
        sets.append(d)
    graphs = {arm: [_graph(arm, d, ctx_frames) for d in sets] for arm in ARMS}
    lanes = {arm: EvaluationLanes(graphs[arm], 8) if arm != "cast" else None for arm in ARMS}
    cast_streams = [torch.cuda.Stream() for _ in range(8)]

    def serial(arm):
        return lambda: [g.graph.replay() for g in graphs[arm]]

    def laned(arm):
        if arm != "cast":
            ln = lanes[arm]

            def run():
                ln.fork()
                for j in range(len(ln)):
                    ln.submit(j)
                ln.join()
            return run
        cur = torch.cuda.current_stream()

        def run_cast():
            for s_ in cast_streams:
                s_.wait_stream(cur)
            for j, g in enumerate(graphs["cast"]):
                with torch.cuda.stream(cast_streams[j % 8]):
                    g.graph.replay()
            for s_ in cast_streams:
                cur.wait_stream(s_)
        return run_cast

    res = {mode: {arm: [] for arm in ARMS} for mode in ("serial", "lanes8")}
    for _ in range(repeats):
        for mode, mk in (("serial", serial), ("lanes8", laned)):
            for arm in ARMS:
                sec = _time(mk(arm), steps)
                res[mode][arm].append(NSETS * steps / sec)
    return res, graphs


def config4(steps, repeats):
    c = {k: v for k, v in CONFIGS["cfg4_batched"].items() if k not in ("nprob", "ctx")}
    P = CONFIGS["cfg4_batched"]["nprob"]
    d = make_inputs(J=8, kind="uniform", seed=5, device="cuda", B=P * c["B"], **{k: v for k, v in c.items() if k != "B"})
    stk = {k: v.reshape(P, c["B"], *v.shape[1:]) for k, v in d.items()}
    stk["real"], stk["fake"] = stk["real"].to(BF), stk["fake"].to(BF)
    hm = [stk[k].requires_grad_(True) for k in INPUT_ORDER[2:]]
    bufs = {"bf16": (stk["real"], stk["fake"]), "fp32": (stk["real"].float(), stk["fake"].float())}

    def run(arm):
        def go():
            if arm == "cast":
                r, f = stk["real"].float(), stk["fake"].float()
            else:
                r, f = bufs[arm]
            f = f.detach().requires_grad_(True)
            loss = gan_utils.compute_sinkhorn_loss_batched(r, f, S, *hm)
            g = torch.autograd.grad(loss.sum(), [f, *hm])
            if arm == "cast":
                g[0].to(BF)
        return go

    res = {arm: [] for arm in ARMS}
    for _ in range(repeats):
        for arm in ARMS:
            res[arm].append(P * steps / _time(run(arm), steps))
    return res, run


def profile(fns, outdir):
    """{label: {kernel: mean us per evaluation}} from torch.profiler, one pass per label"""
    from torch.profiler import ProfilerActivity, profile as tprof
    out = {}
    for label, (fn, nevals) in fns.items():
        fn()
        torch.cuda.synchronize()
        with tprof(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                fn()
            torch.cuda.synchronize()
        ker = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" and e.self_device_time_total > 0:
                ker[e.key[:90]] = round(e.self_device_time_total / (5 * nevals), 2)
        out[label] = dict(sorted(ker.items(), key=lambda kv: -kv[1])[:14])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--no-profile", action="store_true")
    a = ap.parse_args()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        card = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        card = f"nvidia-smi query failed: {e}"
    print("card:", card, flush=True)
    assert _lib.load().kccot_device_check() == 0, _lib.last_error()
    report = {"card": card, "evals_per_s": {}, "gate_cfg2": None}
    prof_fns = {}
    for label, name, ctx in (("cfg1", "cfg1_mmnist", 0), ("cfg2", "cfg2_mazes", 0), ("cfg2_ctx3", "cfg2_mazes", 3)):
        res, graphs = graph_config(name, ctx, a.steps, a.repeats)
        report["evals_per_s"][label] = res
        print(label, json.dumps(res), flush=True)
        for arm in ARMS:
            prof_fns[f"{label}/{arm}"] = ((lambda gs: (lambda: [g.graph.replay() for g in gs]))(graphs[arm]), NSETS)
    res4, run4 = config4(max(2, a.steps // 8), a.repeats)
    report["evals_per_s"]["cfg4"] = {"serial": res4}
    print("cfg4", json.dumps(res4), flush=True)
    P = CONFIGS["cfg4_batched"]["nprob"]
    for arm in ARMS:
        prof_fns[f"cfg4/{arm}"] = (run4(arm), P)
    c2 = report["evals_per_s"]["cfg2"]
    report["gate_cfg2"] = all(min(c2[m]["bf16"]) > max(c2[m]["cast"]) for m in ("serial", "lanes8"))
    print("gate cfg2 (every bf16 run beats every cast run, serial and 8 lanes):", report["gate_cfg2"], flush=True)
    if not a.no_profile:
        report["kernels_us_per_eval"] = profile(prof_fns, a.out)
        for k, v in report["kernels_us_per_eval"].items():
            print(k, json.dumps(v), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bf16_bench.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
