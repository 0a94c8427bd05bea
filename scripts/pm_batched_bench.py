"""Batched martingale penalty against a loop of single-problem calls at the config-4 shape: 256 problems of [64, 10, 8].

    python scripts/pm_batched_bench.py [--steps N] [--obj-steps N] [--repeats R] [--out DIR]

Legs:
    p_M alone, C-ABI calls: forward, backward, forward + backward, each as
        batched    one kccot_pm_batched_fwd / _bwd call over the 256 problems,
        loop       256 kccot_pm_fwd / _bwd calls, problem p with gpm[p];
    the discriminator objective of kernel_train.py:249-250 for 256 problems, forward + autograd.grad w.r.t. m_real,
    h_real, h_fake and m_fake:  (-compute_sinkhorn_loss_batched(...) + p_M).sum(), with p_M
        batched    scale_invariante_martingale_regularization_batched(m_real, ...),
        loop       torch.stack of 256 scale_invariante_martingale_regularization(m_real[p], ...).
Each leg is issued eagerly from Python and replayed as one CUDA graph that holds the same work.  Every leg is warmed up;
the legs alternate inside each of the repeats; times are CUDA events around `steps` calls (the median of the repeats is
printed, all of them are in the JSON).  M is 5.2 MB and stays in L2, as it does in a training step, where the
discriminator has just written it.  The card's name and power limit are read in the same run and printed first.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from batched_smooth_bench import _graph, _time, card  # noqa: E402
from kccotgan_b200 import _lib, gan_utils  # noqa: E402
from kccotgan_b200.functional import _ptr, _stream  # noqa: E402
from kccotgan_b200.synthetic import CONFIGS  # noqa: E402

C4 = CONFIGS["cfg4_batched"]
NPROB, B, T, J = C4["nprob"], C4["B"], C4["T"], 8
VIDEO = tuple(C4[k] for k in ("B", "H", "T", "W", "C"))
LAM, S = 1.0, 1.0 / 15.0


class PmCalls:
    """Buffers of the p_M legs and their C-ABI calls."""

    def __init__(self, M, gpm):
        self.M, self.gpm = M, gpm
        self.pm = torch.empty(NPROB, device="cuda")
        self.stats = torch.empty((NPROB, 2 * J + (T - 1) * J), device="cuda")
        self.gM = torch.empty_like(M)

    def batched(self, d):
        st = _stream(self.M.device)
        if d in ("fwd", "fwd+bwd"):
            _lib.call("kccot_pm_batched_fwd", _ptr(self.M), NPROB, B, T, J, LAM, S, _ptr(self.pm), _ptr(self.stats), st)
        if d in ("bwd", "fwd+bwd"):
            _lib.call("kccot_pm_batched_bwd", _ptr(self.M), NPROB, B, T, J, LAM, S, _ptr(self.stats), _ptr(self.gpm),
                      _ptr(self.gM), st)

    def loop(self, d):
        st = _stream(self.M.device)
        for p in range(NPROB):
            if d in ("fwd", "fwd+bwd"):
                _lib.call("kccot_pm_fwd", _ptr(self.M[p]), B, T, J, LAM, S, _ptr(self.pm[p:]), _ptr(self.stats[p]), st)
            if d in ("bwd", "fwd+bwd"):
                _lib.call("kccot_pm_bwd", _ptr(self.M[p]), B, T, J, LAM, S, _ptr(self.stats[p]), _ptr(self.gpm[p:]),
                          _ptr(self.gM[p]), st)


def _objective_fns(leaves):
    real, fake, h_fake, m_real, h_real, m_fake = leaves
    wrt = [m_real, h_real, h_fake, m_fake]

    def run(pm_fn):
        losses = gan_utils.compute_sinkhorn_loss_batched(real, fake, S, h_fake, m_real, h_real, m_fake)
        return torch.autograd.grad((-losses + pm_fn(m_real)).sum(), wrt)

    def batched():
        return run(lambda m: gan_utils.scale_invariante_martingale_regularization_batched(m, LAM, S))

    def loop():
        return run(lambda m: torch.stack([gan_utils.scale_invariante_martingale_regularization(m[p], LAM, S)
                                          for p in range(NPROB)]))
    return {"batched": batched, "loop": loop}


def _measure(legs, steps, repeats, lib, report, key):
    for leg, fn in legs.items():
        n0 = lib.kccot_launch_count()
        fn()
        report["launches"][f"{key}_{leg}"] = int(lib.kccot_launch_count() - n0)
    graphs = {leg: _graph(fn) for leg, fn in legs.items()}
    runs = {f"{leg}_{how}": [] for leg in legs for how in ("eager", "graph")}
    for _ in range(repeats):
        for leg, fn in legs.items():
            runs[f"{leg}_eager"].append(_time(fn, steps))
            runs[f"{leg}_graph"].append(_time(graphs[leg].replay, steps))
    report["us"][key] = runs
    med = {k: sorted(v)[len(v) // 2] for k, v in runs.items()}
    print(f"  {key:12s} " + "  ".join(f"{k} {t:9.1f} us [{min(runs[k]):.1f}-{max(runs[k]):.1f}]"
                                      for k, t in med.items()), flush=True)
    return med


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="calls per timed window of the p_M legs")
    ap.add_argument("--obj-steps", type=int, default=20, help="calls per timed window of the objective legs")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    lib = _lib.load()
    assert lib.kccot_device_check() == 0, _lib.last_error()
    report = {"card": card(), "nprob": NPROB, "shape": (B, T, J), "video": VIDEO, "steps": a.steps,
              "obj_steps": a.obj_steps, "repeats": a.repeats, "us": {}, "launches": {}}
    print("card:", report["card"], flush=True)
    g = torch.Generator(device="cuda").manual_seed(0)
    M = torch.sigmoid(torch.randn((NPROB, B, T, J), generator=g, device="cuda"))
    gpm = torch.randn(NPROB, generator=g, device="cuda")
    print(f"{NPROB} x [{B}, {T}, {J}]; microseconds per call, median of {a.repeats} [min-max]", flush=True)
    c = PmCalls(M, gpm)
    c.batched("fwd")
    for d in ("fwd", "bwd", "fwd+bwd"):
        _measure({"batched": lambda d=d: c.batched(d), "loop": lambda d=d: c.loop(d)}, a.steps, a.repeats, lib, report,
                 f"pm_{d}")
    # the batched p_M is bit-identical to the loop: the legs time the same numbers
    c.batched("fwd+bwd")
    ref = (c.pm.clone(), c.stats.clone(), c.gM.clone())
    c.loop("fwd+bwd")
    torch.cuda.synchronize()
    assert torch.equal(ref[0], c.pm) and torch.equal(ref[1], c.stats) and torch.equal(ref[2], c.gM)

    vids = [torch.rand((NPROB, *VIDEO), generator=g, device="cuda") for _ in range(2)]
    hm = [torch.sigmoid(torch.randn((NPROB, B, T, J), generator=g, device="cuda")).requires_grad_(True)
          for _ in range(4)]
    fns = _objective_fns(vids + hm)
    ga, gb = fns["batched"](), fns["loop"]()
    torch.cuda.synchronize()
    report["objective_grads_equal"] = all(torch.equal(x, y) for x, y in zip(ga, gb))
    med = _measure(fns, a.obj_steps, a.repeats, lib, report, "objective")
    print(f"objective: the loop adds {med['loop_eager'] - med['batched_eager']:.1f} us eager, "
          f"{med['loop_graph'] - med['batched_graph']:.1f} us graphed; gradients of both legs bit-identical: "
          f"{report['objective_grads_equal']}", flush=True)
    print("launches per call:", json.dumps(report["launches"]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "pm_batched_bench.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
