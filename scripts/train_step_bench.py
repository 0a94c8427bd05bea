"""One kernel_train.py iteration (discriminator step + generator step) with stub networks around the loss
path (kccotgan_b200.train_step), timed end to end with CUDA events: eager and graphed, each at a fixed sigma = 5.0 and
at kernel_train.py's annealed sigma_t = annealing_sigma(5.0, t) (a new float every iteration; the graphed figure
includes the SmoothingTaps.set of every step).

    python scripts/train_step_bench.py cfg3_bair 1d
"""
import sys, os, subprocess
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from kccotgan_b200.data_utils import KernelSmoothing
from kccotgan_b200.synthetic import CONFIGS
from kccotgan_b200.train_step import GraphedTrainingIteration, StubDiscriminator, StubGenerator, make_training_steps

name = sys.argv[1] if len(sys.argv) > 1 else "cfg2_mazes"
kernel = sys.argv[2] if len(sys.argv) > 2 else "none"
c = CONFIGS[name]
B, T, ctx, H, W, C = c["B"], c["T"], c["ctx"], c["H"], c["W"], c["C"]
dev = torch.device("cuda")
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
except OSError:
    power = "unknown"
print(f"device: {torch.cuda.get_device_name(dev)}, power limit {power}")
torch.manual_seed(1)
gen = StubGenerator(T - ctx, C).to(dev)
dh, dm = StubDiscriminator(H, W, C).to(dev), StubDiscriminator(H, W, C).to(dev)
disc_step, gen_step = make_training_steps(gen, dh, dm, B, kernel_choice=kernel)
data = [torch.rand(B, H, T, W, C, device=dev) for _ in range(4)]
anneal = KernelSmoothing().annealing_sigma
n = 20


def timed(fn):
    for i in range(3): fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n): out = fn(i)
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, out


def iteration(i, sigma):
    x = data[i % 4]
    real_in, real_pred = x[:, :, :ctx], x[:, :, ctx:]
    pm = disc_step(real_in, real_pred, sigma)
    return gen_step(real_in, real_pred, sigma), pm


for label, sig in (("sigma 5.0", lambda i: 5.0), ("annealed sigma", lambda i: anneal(5.0, i))):
    ms, (loss, pm) = timed(lambda i: iteration(i, sig(i)))
    print(f"{name} kernel={kernel}, {label}: {ms:.3f} ms per training iteration (disc + gen step, stub nets); "
          f"loss {float(loss):.5f} pM {float(pm):.5f}")

# the same iteration recorded into one CUDA graph
git = GraphedTrainingIteration(gen, dh, dm, data[0][:, :, :ctx], data[0][:, :, ctx:], sigma=5.0, kernel_choice=kernel)
def giter(i, sigma):
    x = data[i % 4]
    git.real_in.copy_(x[:, :, :ctx]); git.real_pred.copy_(x[:, :, ctx:])
    return git.step(sigma)
for rnd in range(3):                  # alternating, so that the spread between rounds shows
    for label, sig in (("sigma 5.0", lambda i: None), ("annealed sigma", lambda i: anneal(5.0, 1000 * rnd + i))):
        ms, (loss, pm) = timed(lambda i: giter(i, sig(i)))
        print(f"{name} kernel={kernel}, {label}: {ms:.3f} ms per GRAPHED training iteration (incl. the copy of the "
              f"batch into the static buffers); loss {float(loss):.5f} pM {float(pm):.5f}")
