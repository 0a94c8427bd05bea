"""bf16 videos in the Gaussian smoothing: three arms on the same inputs at the config-3 shape [64, 64, 12, 64, 3].

    python scripts/bf16_smooth_bench.py [--steps N] [--repeats R] [--out DIR]

Arms:
    fp32      fp32 videos, kccot_smooth_fwd / _bwd;
    bf16      bf16 videos, kccot_smooth_fwd_bf16 / _bwd_bf16;
    cast      bf16 videos through the caller-side route: .float(), the fp32 call, .to(bf16) (and the same around the
              backward), which is what a bf16 caller can do without the bf16 entry points.
Timed:
    passes    forward and backward of 1d and 3d smoothing on their own: C-ABI calls captured in a CUDA graph, one per
              input set;
    step      the config-3 step with 1d (and 3d) smoothing: smoothing of real and fake, the mixed loss, the loss adjoint
              and the smoothing adjoint of fake, one CUDA graph per input set, replayed serially on one stream and on
              8 streams (as EvaluationLanes does).
Six input sets per arm (a bf16 forward touches 6 x 37.7 MB, more than the 126 MB L2 holds), the arms alternate inside
every repeat, three repeats; microseconds per call (passes) and steps per second from CUDA events.  The byte counts per
element are those of the kernels (the tie mask adds 1/8 byte per pass that touches it).  The card name and power limit
are printed first.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kccotgan_b200 import _lib, gan_utils  # noqa: E402
from kccotgan_b200.data_utils import KernelSmoothing  # noqa: E402
from kccotgan_b200.functional import _ptr, _stream, _taps  # noqa: E402
from kccotgan_b200.synthetic import CONFIGS, make_inputs  # noqa: E402

S = 1.0 / 15.0
SIGMA = 5.0
NSETS = 6
ARMS = ("fp32", "bf16", "cast")
BF = torch.bfloat16
SHAPE = tuple(CONFIGS["cfg3_bair"][k] for k in ("B", "H", "T", "W", "C"))
# bytes per element moved by each arm (from the kernels: reads + writes of every pass)
BYTES = {("fwd", "1d"): {"fp32": 12, "bf16": 6 + 1 / 8, "cast": 6 + 12 + 6},
         ("bwd", "1d"): {"fp32": 8 + 12, "bf16": 4 + 1 / 8 + 4 + 1 / 8, "cast": 6 + 20 + 6},
         ("fwd", "3d"): {"fp32": 8 + 8 + 4 + 8, "bf16": 6 + 8 + 4 + 6 + 1 / 8, "cast": 6 + 28 + 6},
         ("bwd", "3d"): {"fp32": 8 + 12 + 8 + 8, "bf16": 4 + 1 / 8 + 6 + 1 / 8 + 8 + 6, "cast": 6 + 36 + 6}}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name()} | {q}"


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
    return a.elapsed_time(b) / 1e3


class Passes:
    """Buffers of one input set and the C-ABI calls of one arm and mode."""

    def __init__(self, arm, mode, x16, g16):
        lib = _lib.load()
        B, H, T, W, C = SHAPE
        self.arm, self.mode = arm, mode
        self.dims = (B, H, T, W, C)
        taps = tuple(KernelSmoothing._weights(3, SIGMA))
        (self.at, self.rt), (self.as_, self.rs) = ((_taps(taps), _taps(None)) if mode == 1 else
                                                   (_taps(None), _taps(taps)))
        dev = x16.device
        self.ws = torch.empty(max(256, lib.kccot_smooth_workspace_bytes(mode, *self.dims)), dtype=torch.uint8,
                              device=dev)
        self.maxval = torch.empty(1, device=dev)
        if arm == "bf16":
            self.x, self.gout = x16, g16
            self.out, self.gx = torch.empty_like(x16), torch.empty_like(x16)
            self.ties = torch.empty(lib.kccot_smooth_ties_bytes(*self.dims) // 4, dtype=torch.int32, device=dev)
        else:
            self.x, self.gout = x16.float(), g16.float()
            self.out, self.gx = torch.empty_like(self.x), torch.empty_like(self.x)
            if arm == "cast":
                self.x16, self.g16 = x16, g16
                self.out16, self.gx16 = torch.empty_like(x16), torch.empty_like(x16)

    def fwd(self):
        if self.arm == "bf16":
            _lib.call("kccot_smooth_fwd_bf16", self.mode, _ptr(self.x), *self.dims, self.at, self.rt, self.as_, self.rs,
                      _ptr(self.out), _ptr(self.maxval), _ptr(self.ties), _ptr(self.ws), self.ws.numel(),
                      _stream(self.x.device))
            return
        if self.arm == "cast":
            self.x.copy_(self.x16)
        _lib.call("kccot_smooth_fwd", self.mode, _ptr(self.x), *self.dims, self.at, self.rt, self.as_, self.rs,
                  _ptr(self.out), _ptr(self.maxval), _ptr(self.ws), self.ws.numel(), _stream(self.x.device))
        if self.arm == "cast":
            self.out16.copy_(self.out)

    def bwd(self):
        if self.arm == "bf16":
            _lib.call("kccot_smooth_bwd_bf16", self.mode, _ptr(self.gout), _ptr(self.out), _ptr(self.maxval),
                      _ptr(self.ties), *self.dims, self.at, self.rt, self.as_, self.rs, _ptr(self.gx), _ptr(self.ws),
                      self.ws.numel(), _stream(self.x.device))
            return
        if self.arm == "cast":
            self.gout.copy_(self.g16)
        _lib.call("kccot_smooth_bwd", self.mode, _ptr(self.gout), _ptr(self.out), _ptr(self.maxval), *self.dims,
                  self.at, self.rt, self.as_, self.rs, _ptr(self.gx), _ptr(self.ws), self.ws.numel(),
                  _stream(self.x.device))
        if self.arm == "cast":
            self.gx16.copy_(self.gx)


def bench_passes(sets, steps, repeats):
    res = {}
    for mode, tag in ((1, "1d"), (3, "3d")):
        objs = {arm: [Passes(arm, mode, x, g) for x, g in sets] for arm in ARMS}
        for o in objs.values():
            for p in o:
                p.fwd()
        graphs = {(arm, d): _graph(lambda arm=arm, d=d: [getattr(p, d)() for p in objs[arm]])
                  for arm in ARMS for d in ("fwd", "bwd")}
        for d in ("fwd", "bwd"):
            res[f"{d}_{tag}"] = {arm: [] for arm in ARMS}
        for _ in range(repeats):
            for d in ("fwd", "bwd"):
                for arm in ARMS:
                    sec = _time(graphs[(arm, d)].replay, steps)
                    res[f"{d}_{tag}"][arm].append(sec / (steps * NSETS) * 1e6)
        del objs, graphs
        torch.cuda.empty_cache()
    return res


def _step(arm, d, kernel):
    ks = KernelSmoothing(6, 6)
    smooth = ks.temporal_convolution if kernel == "1d" else ks.gaussian_convolution3D
    real, fake = d["real"], d["fake"]
    if arm == "fp32":
        real, fake = real.float(), fake.float()
    fake = fake.detach().clone().requires_grad_(True)
    hm = [d[k].detach().clone().requires_grad_(True) for k in ("h_fake", "m_real", "h_real", "m_fake")]

    def run():                          # (the current stream: the capture stream inside torch.cuda.graph)
        if arm == "cast":
            rs, fs = smooth(real.float(), SIGMA).to(BF), smooth(fake.float(), SIGMA).to(BF)
        else:
            rs, fs = smooth(real, SIGMA), smooth(fake, SIGMA)
        loss = gan_utils.compute_sinkhorn_loss(rs, fs, S, 0.8, 100, *hm)
        return torch.autograd.grad(loss, [fake, *hm])
    return _graph(run), (real, fake, hm)        # the graph reads these buffers: they must outlive it


def bench_step(inputs, kernel, steps, repeats):
    graphs = {arm: [_step(arm, d, kernel) for d in inputs] for arm in ARMS}
    streams = [torch.cuda.Stream() for _ in range(8)]

    def serial(arm):
        return lambda: [g.replay() for g, _ in graphs[arm]]

    def lanes(arm):
        def run():
            cur = torch.cuda.current_stream()
            for s_ in streams:
                s_.wait_stream(cur)
            for j, (g, _) in enumerate(graphs[arm]):
                with torch.cuda.stream(streams[j % 8]):
                    g.replay()
            for s_ in streams:
                cur.wait_stream(s_)
        return run

    res = {m: {arm: [] for arm in ARMS} for m in ("serial", "lanes8")}
    for _ in range(repeats):
        for m, mk in (("serial", serial), ("lanes8", lanes)):
            for arm in ARMS:
                res[m][arm].append(len(inputs) * steps / _time(mk(arm), steps))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    assert _lib.load().kccot_device_check() == 0, _lib.last_error()
    report = {"card": card(), "shape": SHAPE, "sigma": SIGMA, "nsets": NSETS, "steps": a.steps, "repeats": a.repeats}
    print("card:", report["card"], flush=True)
    g = torch.Generator().manual_seed(0)
    sets = [(torch.rand(SHAPE, generator=g).to(BF).cuda(), torch.randn(SHAPE, generator=g).to(BF).cuda())
            for _ in range(NSETS)]
    passes = bench_passes(sets, a.steps, a.repeats)
    report["passes_us"] = passes
    report["bytes_per_element"] = {f"{d}_{k}": v for (d, k), v in BYTES.items()}
    n = 1
    for v in SHAPE:
        n *= v
    print(f"\nper call, microseconds (median of {a.repeats}; effective TB/s from the byte counts)", flush=True)
    for key, arms in passes.items():
        d, k = key.split("_")
        cells = []
        for arm in ARMS:
            t = sorted(arms[arm])[len(arms[arm]) // 2]
            cells.append(f"{arm} {t:7.1f} us ({BYTES[(d, k)][arm] * n / t / 1e6:4.2f} TB/s)")
        print(f"  {key:7s} " + "  ".join(cells), flush=True)
    del sets
    torch.cuda.empty_cache()
    c = {k: v for k, v in CONFIGS["cfg3_bair"].items() if k not in ("nprob", "ctx")}
    inputs = []
    for i in range(NSETS):
        d = make_inputs(J=8, kind="uniform", seed=1 + 1000 * i, device="cuda", **c)
        d["real"], d["fake"] = d["real"].to(BF), d["fake"].to(BF)
        inputs.append(d)
    report["step_per_s"] = {}
    for kernel in ("1d", "3d"):
        r = bench_step(inputs, kernel, max(1, a.steps // 5), a.repeats)
        report["step_per_s"][kernel] = r
        for m, arms in r.items():
            print(f"  step {kernel} {m:7s} " + "  ".join(f"{arm} {sorted(v)[len(v) // 2]:8.1f}/s" for arm, v in
                                                        arms.items()), flush=True)
    gate = all(max(v["bf16"]) < min(v["cast"]) for v in passes.values())
    gate = gate and all(min(arms["bf16"]) > max(arms["cast"]) for r in report["step_per_s"].values()
                        for arms in r.values())
    report["bf16_beats_cast_everywhere"] = gate
    print("every bf16 run beats every cast run, on every arm:", gate, flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bf16_smooth_bench.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
