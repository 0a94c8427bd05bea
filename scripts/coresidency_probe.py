"""Co-residency probe (config 2 shapes): do two streaming kernels of different evaluations share SMs?

    python scripts/coresidency_probe.py [N] [STEPS]

Part 1 calls the C ABI as bench.py::stage_times does and times, with CUDA events:
    N back-to-back kccot_mixed_sqdist_partials on one stream,
    N back-to-back kccot_mixed_cost_bwd (gradient of the fake rows only: W' image + gradient GEMM) on one stream,
and the same launches split over two streams (sqdist || gradient, gradient || gradient, sqdist || sqdist).
If CTAs of the two streams share SMs, the two-stream time is clearly below the sum of the one-stream times;
if every kernel needs a whole SM, the two-stream time is about the sum.
Part 2 is the EvaluationLanes sweep over 1 / 2 / 4 / 8 / 12 lanes (as scripts/overlap_probe.py).
The card name, power limit and maximum SM clock are printed first (an nvidia-smi query).
"""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kccotgan_b200 import _lib  # noqa: E402
from kccotgan_b200 import functional as F  # noqa: E402
from kccotgan_b200.graphed import EvaluationLanes, GraphedSinkhornLoss  # noqa: E402
from kccotgan_b200.synthetic import CONFIGS, INPUT_ORDER, make_inputs  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 200
STEPS = int(sys.argv[2]) if len(sys.argv) > 2 else 1200
S = 1.0 / 15.0
J = 8
NSETS = 12

try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    print("card:", q.stdout.strip() or q.stderr.strip(), flush=True)
except (OSError, subprocess.TimeoutExpired) as e:
    print("card: nvidia-smi query failed:", e, flush=True)

dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
lib = _lib.load()
cfg = {k: v for k, v in CONFIGS["cfg2_mazes"].items() if k != "nprob"}
B, T = cfg["B"], cfg["T"]
sets = [make_inputs(J=J, kind="uniform", seed=1 + 1000 * i, device=dev, **cfg) for i in range(NSETS)]
K = sets[0]["real"][0].numel()
p = F._ptr


class Lane:
    """Workspaces and outputs of one stream: nothing is shared between the two streams."""

    def __init__(self):
        self.stream = torch.cuda.Stream(dev)
        self.ws = torch.empty(lib.kccot_mixed_cost_workspace_bytes(1, B, K), dtype=torch.uint8, device=dev)
        self.ws3 = torch.empty(lib.kccot_mixed_cost_bwd_workspace_bytes(1, B, K), dtype=torch.uint8, device=dev)
        self.Cb = torch.randn(3, B, B, device=dev) * 1e-3
        self.gf = torch.empty(B, K, device=dev)
        with torch.cuda.stream(self.stream):
            self.st = F._stream(dev)          # raw handle for the C ABI

    def views(self, i):
        d = sets[i % NSETS]
        return [d[k].detach() for k in INPUT_ORDER]

    def sqdist(self, i):
        r, f = self.views(i)[:2]
        _lib.call("kccot_mixed_sqdist_partials", p(r.reshape(B, -1)), p(f.reshape(B, -1)), 1, B, K, p(self.ws),
                  self.ws.numel(), 0, self.st)

    def grad(self, i):
        r, f, hf, mr, hr, mf = self.views(i)
        _lib.call("kccot_mixed_cost_bwd", p(self.Cb), p(r.reshape(B, -1)), p(f.reshape(B, -1)), 1, B, K, p(hf), p(mr),
                  p(hr), p(mf), T, J, S, None, p(self.gf), None, None, None, None, p(self.ws3), self.ws3.numel(), 0,
                  self.st)


lanes = [Lane(), Lane()]


def timed(jobs, n):
    """jobs: list of (lane, fn name); job j issues n launches on its lane, input sets rotating (cold in L2)."""
    main = torch.cuda.current_stream(dev)
    for warm in (True, False):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        for ln, _ in jobs:
            ln.stream.wait_stream(main)
        for i in range(3 if warm else n):
            for j, (ln, fn) in enumerate(jobs):
                getattr(ln, fn)(i + 5 * j)
        for ln, _ in jobs:
            main.wait_stream(ln.stream)
        e1.record(main)
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n      # us per launch round


a, b = lanes
t_sq = timed([(a, "sqdist")], N)
t_gr = timed([(a, "grad")], N)
print(f"one stream:  sqdist {t_sq:6.2f} us   gradient (W' image + GEMM) {t_gr:6.2f} us per call", flush=True)
for name, jobs, alone in (("sqdist || gradient", [(a, "sqdist"), (b, "grad")], t_sq + t_gr),
                          ("gradient || gradient", [(a, "grad"), (b, "grad")], 2 * t_gr),
                          ("sqdist || sqdist", [(a, "sqdist"), (b, "sqdist")], 2 * t_sq)):
    t = timed(jobs, N)
    print(f"two streams, {name:22s}: {t:6.2f} us per pair, sum of one-stream times {alone:6.2f} us "
          f"({t / alone:5.3f} of the sum)", flush=True)

# ---- EvaluationLanes sweep ---------------------------------------------------------------------------------------
del lanes, a, b
graphs = [GraphedSinkhornLoss(*[d[k] for k in INPUT_ORDER], S, adopt=True) for d in sets]
torch.cuda.synchronize()
ref = []
for g in graphs:
    g.step()
    torch.cuda.synchronize()
    ref.append((float(g.loss.detach()), g.grads["fake"].clone()))
for nl in (1, 2, 4, 8, 12):
    lanes = EvaluationLanes(graphs, nl)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for n in (60, STEPS):
        torch.cuda.synchronize()
        e0.record()
        lanes.fork()
        for i in range(n):
            lanes.submit(i % NSETS)
        lanes.join()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    ok = all(float(g.loss.detach()) == r[0] and torch.equal(g.grads["fake"], r[1]) for g, r in zip(graphs, ref))
    print(f"{nl:2d} lane(s): {STEPS / ms * 1e3:8.0f} evals/s ({ms / STEPS * 1e3:6.2f} us per evaluation), "
          f"results identical to serial replays: {ok}", flush=True)
