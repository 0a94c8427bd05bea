"""Batched smoothing against a loop of single-problem calls at the config-4 shape: 256 problems of [64, 32, 10, 32, 1].

    python scripts/batched_smooth_bench.py [--steps N] [--repeats R] [--out DIR]

Legs, for fp32 and bf16 videos, modes 1 (temporal) and 3 (3-D), forward and backward:
    batched        one kccot_smooth_batched_* call over the 256 problems;
    loop           256 calls of the single-problem *_dev entries, problem p with weights row p;
each issued eagerly from Python and replayed as a CUDA graph that holds the same calls.  Every leg is warmed up; the
legs alternate inside each of the repeats; times are CUDA events around `steps` calls.  A batch (671 MB in fp32, 336 MB
in bf16) is larger than the 126 MB L2, so every call streams from HBM.  The bytes per element are those the passes move
(reads and writes of every pass; the bf16 tie mask adds 1/8 byte to each pass that touches it), and the achieved rate is
those bytes over the measured time.  The card's name and power limit are read in the same run and printed first.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kccotgan_b200 import _lib  # noqa: E402
from kccotgan_b200.data_utils import KernelSmoothing, SmoothingTaps  # noqa: E402
from kccotgan_b200.functional import _ptr, _stream  # noqa: E402
from kccotgan_b200.synthetic import CONFIGS  # noqa: E402

C4 = CONFIGS["cfg4_batched"]
NPROB = C4["nprob"]
SHAPE = tuple(C4[k] for k in ("B", "H", "T", "W", "C"))
RADIUS = 3
BF = torch.bfloat16
# bytes per element moved by the passes of each call (reads + writes)
BYTES = {("fwd", 1): {"fp32": 12, "bf16": 6 + 1 / 8},
         ("bwd", 1): {"fp32": 8 + 12, "bf16": 4 + 1 / 8 + 4 + 1 / 8},
         ("fwd", 3): {"fp32": 8 + 8 + 4 + 8, "bf16": 6 + 8 + 4 + 6 + 1 / 8},
         ("bwd", 3): {"fp32": 8 + 12 + 8 + 8, "bf16": 4 + 1 / 8 + 6 + 1 / 8 + 8 + 6}}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name()} | {q}"


class Calls:
    """Buffers of one dtype and mode, and the C-ABI calls of both legs."""

    def __init__(self, dtype, mode, x, gout, taps):
        lib = _lib.load()
        self.mode, self.bf16 = mode, dtype == BF
        self.x, self.gout = x.to(dtype), gout.to(dtype)
        self.out, self.gx = torch.empty_like(self.x), torch.empty_like(self.x)
        self.w = taps.weights
        self.maxval = torch.empty(NPROB, device="cuda")
        self.ws = torch.empty(lib.kccot_smooth_batched_workspace_bytes(mode, NPROB, *SHAPE), dtype=torch.uint8,
                              device="cuda")
        self.ws1 = torch.empty(max(256, lib.kccot_smooth_workspace_bytes(mode, *SHAPE)), dtype=torch.uint8,
                               device="cuda")
        self.ties = torch.empty(lib.kccot_smooth_ties_bytes(NPROB * SHAPE[0], *SHAPE[1:]) // 4, dtype=torch.int32,
                                device="cuda")
        self.n = self.x[0].numel()
        assert self.n % 32 == 0                 # problem p's tie words are a slice of the batch's mask
        self.sfx = "_bf16" if self.bf16 else ""

    def batched(self, d):
        st = _stream(self.x.device)
        dims = (NPROB, *SHAPE)
        tie = (_ptr(self.ties),) if self.bf16 else ()
        if d == "fwd":
            _lib.call("kccot_smooth_batched_fwd" + self.sfx, self.mode, _ptr(self.x), *dims, _ptr(self.w), RADIUS,
                      _ptr(self.out), _ptr(self.maxval), *tie, _ptr(self.ws), self.ws.numel(), st)
        else:
            _lib.call("kccot_smooth_batched_bwd" + self.sfx, self.mode, _ptr(self.gout), _ptr(self.out),
                      _ptr(self.maxval), *tie, *dims, _ptr(self.w), RADIUS, _ptr(self.gx), _ptr(self.ws),
                      self.ws.numel(), st)

    def loop(self, d):
        st = _stream(self.x.device)
        for p in range(NPROB):
            tie = (_ptr(self.ties[p * self.n // 32:]),) if self.bf16 else ()
            if d == "fwd":
                _lib.call("kccot_smooth_fwd" + self.sfx + "_dev", self.mode, _ptr(self.x[p]), *SHAPE, _ptr(self.w[p]),
                          RADIUS, _ptr(self.out[p]), _ptr(self.maxval[p:]), *tie, _ptr(self.ws1), self.ws1.numel(), st)
            else:
                _lib.call("kccot_smooth_bwd" + self.sfx + "_dev", self.mode, _ptr(self.gout[p]), _ptr(self.out[p]),
                          _ptr(self.maxval[p:]), *tie, *SHAPE, _ptr(self.w[p]), RADIUS, _ptr(self.gx[p]),
                          _ptr(self.ws1), self.ws1.numel(), st)


def _graph(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def _time(fn, steps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / steps          # microseconds per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    lib = _lib.load()
    assert lib.kccot_device_check() == 0, _lib.last_error()
    report = {"card": card(), "nprob": NPROB, "shape": SHAPE, "radius": RADIUS, "steps": a.steps,
              "repeats": a.repeats, "bytes_per_element": {f"{d}_{m}": v for (d, m), v in BYTES.items()}, "us": {},
              "launches": {}}
    print("card:", report["card"], flush=True)
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand((NPROB, *SHAPE), generator=g, device="cuda")
    gout = torch.randn((NPROB, *SHAPE), generator=g, device="cuda")
    ks = KernelSmoothing()
    taps = SmoothingTaps(RADIUS, nprob=NPROB).set([ks.annealing_sigma(5.0, 40 * p) for p in range(NPROB)])
    elems = NPROB * x[0].numel()
    print(f"{NPROB} x {list(SHAPE)}, radius {RADIUS}; microseconds per call (median of {a.repeats}), achieved TB/s "
          "from the bytes the passes move", flush=True)
    for dtype, dname in ((torch.float32, "fp32"), (BF, "bf16")):
        for mode in (1, 3):
            c = Calls(dtype, mode, x, gout, taps)
            c.batched("fwd")
            for d in ("fwd", "bwd"):
                legs = {"batched": lambda d=d: c.batched(d), "loop": lambda d=d: c.loop(d)}
                for leg, fn in legs.items():
                    n0 = lib.kccot_launch_count()
                    fn()
                    report["launches"][f"{dname}_mode{mode}_{d}_{leg}"] = int(lib.kccot_launch_count() - n0)
                graphs = {leg: _graph(fn) for leg, fn in legs.items()}
                runs = {f"{leg}_{how}": [] for leg in legs for how in ("eager", "graph")}
                for _ in range(a.repeats):
                    for leg, fn in legs.items():
                        runs[f"{leg}_eager"].append(_time(fn, a.steps))
                        runs[f"{leg}_graph"].append(_time(graphs[leg].replay, a.steps))
                key = f"{dname}_mode{mode}_{d}"
                report["us"][key] = runs
                nbytes = BYTES[(d, mode)][dname] * elems
                cells = []
                for k, v in runs.items():
                    t = sorted(v)[len(v) // 2]
                    cells.append(f"{k} {t:9.1f} us ({nbytes / t / 1e6:4.2f} TB/s)")
                print(f"  {key:16s} " + "  ".join(cells), flush=True)
                del graphs
            del c
            torch.cuda.empty_cache()
    print("launches per call:", json.dumps(report["launches"]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "batched_smooth_bench.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
