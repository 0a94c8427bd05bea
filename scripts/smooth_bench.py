"""Times the smoothing kernels (KernelSmoothing.temporal_convolution / gaussian_convolution3D, forward and
backward) at BASELINE config 3's video shape; prints us and GB/s against the algorithmic bytes.  Each pass runs with
host weights (a float sigma: kccot_smooth_fwd / _bwd) and with device weights (a SmoothingTaps: the *_dev entries,
which read the weights as the kernels start), alternating, so that any cost of the weight read shows."""
import sys, os, subprocess
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from kccotgan_b200 import _lib, functional as F
from kccotgan_b200.data_utils import KernelSmoothing, SmoothingTaps
from kccotgan_b200.synthetic import CONFIGS

c = CONFIGS["cfg3_bair"]
B, T, H, W, C = c["B"], c["T"], c["H"], c["W"], c["C"]
nbytes = B * T * H * W * C * 4
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
except OSError:
    power = "unknown"
print(f"device: {torch.cuda.get_device_name()}, power limit {power}")
ks = KernelSmoothing(temporal_kernel_size=6, spatial_kernel_size=6)
taps = SmoothingTaps(3).set(5.0)
xs = [torch.rand(B, H, T, W, C, device="cuda").requires_grad_(True) for _ in range(6)]     # rotate: 6 x 151 MB > L2
def timeit(fn, reps=30):
    for i in range(3): fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps): fn(i)
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3
lib = _lib.load()
dev = xs[0].device
p = F._ptr
for name, op in (("temporal_convolution", ks.temporal_convolution), ("gaussian_convolution3D", ks.gaussian_convolution3D)):
    gs = [torch.rand_like(x) for x in xs]
    # the same C-ABI calls captured in CUDA graphs (no Python / launch gaps; input L2-resident)
    mode = 1 if name == "temporal_convolution" else 3
    htaps, rad = F._taps(tuple(ks._weights(3, 5.0)))
    weights = {"float sigma": (htaps, rad, htaps, rad), "SmoothingTaps": (p(taps.weights), rad)}
    x0 = xs[0].detach(); g0 = gs[0]
    o0 = torch.empty_like(x0); gx0 = torch.empty_like(x0); mx = torch.empty(1, device=dev)
    wsb = torch.empty(lib.kccot_smooth_workspace_bytes(mode, B, H, T, W, C), dtype=torch.uint8, device=dev)
    graphs = {}
    for label, sfx in (("float sigma", ""), ("SmoothingTaps", "_dev")):
        def fwd_abi():
            _lib.call("kccot_smooth_fwd" + sfx, mode, p(x0), B, H, T, W, C, *weights[label], p(o0), p(mx), p(wsb),
                      wsb.numel(), F._stream(dev))
        def bwd_abi():
            _lib.call("kccot_smooth_bwd" + sfx, mode, p(g0), p(o0), p(mx), B, H, T, W, C, *weights[label], p(gx0),
                      p(wsb), wsb.numel(), F._stream(dev))
        fwd_abi(); bwd_abi(); torch.cuda.synchronize()
        gf, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(gf):
            fwd_abi()
        with torch.cuda.graph(gb):
            bwd_abi()
        graphs[label] = (gf, gb)
    for rnd in range(3):              # alternating
        for label, sig in (("float sigma", 5.0), ("SmoothingTaps", taps)):
            tf = timeit(lambda i: op(xs[i % 6], sig))
            outs = [op(x, sig) for x in xs]
            tb = timeit(lambda i: torch.autograd.grad(outs[i % 6], xs[i % 6], gs[i % 6], retain_graph=True))
            del outs
            gf, gb = graphs[label]
            tgf = timeit(lambda i: gf.replay()); tgb = timeit(lambda i: gb.replay())
            print(f"{name} [{label}]: graph replay fwd {tgf:.1f} us, bwd {tgb:.1f} us (input L2-resident)")
            print(f"{name} [{label}]: tensor {nbytes / 1e6:.1f} MB; fwd {tf:.1f} us ({2 * nbytes / tf / 1e3:.0f} GB/s on "
                  f"read+write), bwd {tb:.1f} us ({2 * nbytes / tb / 1e3:.0f} GB/s on read+write)")
