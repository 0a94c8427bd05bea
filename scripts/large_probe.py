"""Stage timings of the large-batch path through the C ABI (development probe, not a bench line).

    python scripts/large_probe.py [B K [reps]]

Prints ms and algorithmic TFLOP/s of: mixed cost forward (pre-pass + GEMM + finalize), Sinkhorn forward,
Sinkhorn backward, mixed cost backward (W' build + transposed split + GEMM + martingale adjoint); checks a
256 x 256 corner of C_xy against the CUDA-core direct-form kernels.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kccotgan_b200 import _lib, functional as F  # noqa: E402

S = 1.0 / 15.0


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
    K = int(sys.argv[2]) if len(sys.argv) > 2 else 16384
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
    T, J, L = 20, 8, 100
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(1)
    real = torch.rand((B, K), generator=g, device=dev)
    fake = torch.rand((B, K), generator=g, device=dev)
    hm = [torch.sigmoid(torch.randn((B, T, J), generator=g, device=dev)) for _ in range(4)]
    C3 = torch.empty(3, B, B, device=dev)
    Cb = torch.empty_like(C3)
    ws = torch.empty(lib.kccot_mixed_loss_workspace_bytes(1, B, K, L), dtype=torch.uint8, device=dev)
    uh = torch.empty(3, L + 1, B, device=dev)
    vh = torch.empty_like(uh)
    nits = torch.empty(3, dtype=torch.int32, device=dev)
    cost = torch.empty(3, device=dev)
    g3 = torch.tensor([2.0, -1.0, -1.0], device=dev)
    gf = torch.empty(B, K, device=dev)
    gh = [torch.empty(B, T, J, device=dev) for _ in range(4)]
    st = F._stream(dev)
    p = F._ptr
    print(f"B={B} K={K}: workspace {ws.numel() / 1e9:.2f} GB", flush=True)

    def cost_fwd():
        _lib.call("kccot_mixed_cost_fwd", p(real), p(fake), 1, B, K, p(hm[0]), p(hm[1]), p(hm[2]), p(hm[3]), T, J, S,
                  p(C3), p(ws), ws.numel(), 0, st)

    def sk_fwd():
        _lib.call("kccot_sinkhorn_fwd", p(C3), 3, B, 1.0, L, 100, 1e-2, 0, p(uh), p(vh), p(nits), p(cost), p(ws),
                  ws.numel(), st)

    def sk_bwd():
        _lib.call("kccot_sinkhorn_bwd", p(C3), 3, B, 1.0, L, p(uh), p(vh), p(nits), p(g3), p(Cb), p(ws), ws.numel(), st)

    def cost_bwd():
        _lib.call("kccot_mixed_cost_bwd", p(Cb), p(real), p(fake), 1, B, K, p(hm[0]), p(hm[1]), p(hm[2]), p(hm[3]), T, J,
                  S, None, p(gf), p(gh[0]), p(gh[1]), p(gh[2]), p(gh[3]), p(ws), ws.numel(), 0, st)

    flops = {"cost_fwd": 6.0 * B * B * K, "sinkhorn_fwd": None, "sinkhorn_bwd": None, "cost_bwd": 4.0 * B * B * K}
    total = 0.0
    for name, fn in (("cost_fwd", cost_fwd), ("sinkhorn_fwd", sk_fwd), ("sinkhorn_bwd", sk_bwd), ("cost_bwd", cost_bwd)):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        total += ms
        extra = f"  {flops[name] / ms / 1e9:.1f} algorithmic TFLOP/s" if flops[name] else ""
        print(f"{name:14s} {ms:9.3f} ms{extra}", flush=True)
    print(f"eval total     {total:9.3f} ms  -> {1e3 / total:.2f} evals/s, {10.0 * B * B * K / total / 1e9:.1f} algorithmic TFLOP/s",
          flush=True)
    print("loss terms", cost.tolist(), "nits", nits.tolist(), "finite grads", bool(torch.isfinite(gf).all()))

    # corner check against the direct-form CUDA-core kernels
    n = min(256, B)
    Cc = torch.empty(n, n, device=dev)
    wsc = torch.empty(lib.kccot_cost_workspace_bytes(1, n, n, K), dtype=torch.uint8, device=dev)
    r, f = real[:n].contiguous(), fake[:n].contiguous()
    h0, m1 = hm[0][:n].contiguous(), hm[1][:n].contiguous()
    _lib.call("kccot_cost_fwd", p(r), p(f), 1, n, n, K, p(h0), p(m1), None, None, T, J, S, p(Cc), p(wsc), wsc.numel(), 1, st)
    err = (C3[0, :n, :n] - Cc).abs().max() / Cc.abs().max()
    print(f"C_xy corner vs direct form: max rel err {float(err):.2e}")


if __name__ == "__main__":
    main()
