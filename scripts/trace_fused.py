"""Print the cycle timeline of the fused step kernel (MINPPO_TRACE=1) for a few CTAs of the last minibatch step."""
import os, sys
os.environ["MINPPO_TRACE"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import numpy as np, torch
import bench
from minppo_b200 import _lib
from minppo_b200.learner import Learner, Memory, TrainState
from oracle import ppo_numpy as P
from tests.helpers import hyper_to_config

dev = torch.device("cuda:0")
w_ = bench.workload(1)
if os.environ.get("TRACE_ENVS"):                      # probe: fewer (tile, net) CTAs in flight (contention for the shared weights?)
    w_ = dict(w_, num_envs=int(os.environ["TRACE_ENVS"]))
shape = bench.make_shape(w_)
hp = bench.make_hyper(shape)
learner = Learner(hyper_to_config(hp, use_graph=False), bench.OBS_DIM, bench.ACT_DIM, dev)
params, traj, last_val = bench.synth_shard(shape, 0, 1)
t = lambda x: torch.as_tensor(np.ascontiguousarray(x)).to(dev)
mem = Memory(done=t(traj["done"]), action=t(traj["action"]), value=t(traj["value"]), reward=t(traj["reward"]),
             log_prob=t(traj["log_prob"]), obs=t(traj["obs"]))
ts = TrainState.create(P.flatten_params(params, hp.num_layers), dev)
rng = torch.tensor([0, 1337], dtype=torch.int32, device=dev)
for _ in range(2):
    learner.update(ts, mem, t(last_val), rng)
learner.check()
n = 2 * (hp.minibatch_size // 128)
out = torch.empty((n, 256), dtype=torch.int64, device=dev)
_lib.check(learner.lib.minppo_ctx_read(learner._h, 7, out.data_ptr(), out.numel() * 8, torch.cuda.current_stream(dev).cuda_stream))
torch.cuda.synchronize()
tr = out.cpu().numpy()
names = {26: "w: gather issued", 27: "w: loss inputs requested", 28: "w: griddep wait passed", 29: "w: staging loads issued", 30: "w: staging stored", 31: "w: all X blocks published", 16: "kernel start (t0)", 0: "workers start", 1: "gather+stage done, xfull", 17: "mma: start", 18: "mma: X block 0 seen", 19: "mma: L1 issued",
         2: "w: acc0 ready", 3: "w: epi1 done (h1r)", 20: "mma: h1r seen", 21: "mma: L2 issued", 4: "w: acc1 ready", 5: "w: epi2 done (h2r)",
         24: "mma: head fwd issued", 6: "w: head out ready", 7: "w: loss done + tile sums", 25: "mma: dA2/dW2 issued", 8: "w: bwd accs ready",
         9: "w: dz2 epilogue done (dz2r)", 22: "mma: dz2r seen", 23: "mma: dH1 issued", 10: "w: dh1 acc ready", 11: "w: epi3 done", 12: "w: stores done"}
order = [16, 0, 17, 26, 28, 31, 30, 1, 18, 19, 2, 3, 21, 4, 5, 24, 6, 7, 25, 8, 9, 23, 10, 11, 12]
for cta in (0, 1, n // 2, n - 1):
    t0 = tr[cta, 16]
    print(f"--- CTA {cta} ({'actor' if cta < n // 2 else 'critic'})")
    prev = 0
    for k in order:
        d = int(tr[cta, k] - t0)
        print(f"  {names[k]:34s} {d:8d}  (+{d - prev})")
        prev = d
    print("  dH1 GEMM, MMA issuer: k-block seen", [int(tr[cta, 64 + k] - t0) for k in range(4)], "| stage landed", [int(tr[cta, 68 + k] - t0) for k in range(8)],
          "| MMAs issued", [int(tr[cta, 76 + k] - t0) for k in range(8)])
    # every worker warp around the four big epilogues (warp w: lane quadrant w & 3 = scheduler, column share w >> 2)
    for e, nm in enumerate(("epilogue 1 (H1)", "epilogue 2 (H2)", "dZ2 epilogue", "epilogue 3 (dZ1)")):
        st = tr[cta, 128 + 32 * e:128 + 32 * e + 16] - t0
        en = tr[cta, 128 + 32 * e + 16:128 + 32 * e + 32] - t0
        print(f"  {nm:18s} window {int(en.max() - st.min()):5d}  median warp {int(np.median(en - st)):5d}  start {int(st.min())}..{int(st.max())}  end per warp {[int(x) for x in en]}")
for e, nm in enumerate(("epilogue 1 (H1)", "epilogue 2 (H2)", "dZ2 epilogue", "epilogue 3 (dZ1)")):
    st = tr[:, 128 + 32 * e:128 + 32 * e + 16] - tr[:, 16:17]
    en = tr[:, 128 + 32 * e + 16:128 + 32 * e + 32] - tr[:, 16:17]
    late = en - np.median(en, axis=1, keepdims=True)
    for lo, hi, who in ((0, n // 2, "actor"), (n // 2, n, "critic")):
        print(f"{nm:18s} {who:6s} CTAs: window mean {(en[lo:hi].max(axis=1) - st[lo:hi].min(axis=1)).mean():6.0f}  median-warp time {np.median(en[lo:hi] - st[lo:hi], axis=1).mean():6.0f}  "
              f"warps > 1000 cycles behind their CTA's median, per warp id: {(late[lo:hi] > 1000).sum(axis=0).tolist()}")
tot = tr[:, 12] - tr[:, 16]
print("total cycles per CTA: actor mean", tot[:n // 2].mean(), "critic mean", tot[n // 2:].mean(), "max", tot.max())

# ---- dwopt kernel phases (last minibatch step): stamps 0 start, 1 phase-1 done, 2 the CTA's last split-K counter wait
# satisfied (= 1 if it had none), 3 phase-2 done, 4 grid barrier passed, 5 end
nsm = torch.cuda.get_device_properties(dev).multi_processor_count
o2 = torch.empty((nsm, 16), dtype=torch.int64, device=dev)
_lib.check(learner.lib.minppo_ctx_read(learner._h, 8, o2.data_ptr(), o2.numel() * 8, torch.cuda.current_stream(dev).cuda_stream))
torch.cuda.synchronize()
t2 = o2.cpu().numpy()
d = t2[:, 1:6] - t2[:, 0:5]
lab = ["phase1 (GEMM / small leaves)", "counter waits (to last)", "phase 2 (after last wait)", "grid barrier wait", "phase 3 (Adam)"]
print("--- dwopt kernel, cycles per CTA (globaltimer-free: per-SM clock64 deltas)")
for k in range(5):
    print(f"  {lab[k]:30s} gemm CTAs: mean {d[:128, k].mean():8.0f} min {d[:128, k].min():8.0f} max {d[:128, k].max():8.0f}"
          f" | extra CTAs: mean {d[128:, k].mean():8.0f} max {d[128:, k].max():8.0f}")
for gi in range(4):
    seg = d[32 * gi:32 * gi + 32, 0]
    print(f"  phase 1 of GEMM group {gi} (net {gi // 2}, layer {gi % 2}): mean {seg.mean():8.0f} min {seg.min():8.0f} max {seg.max():8.0f}")
print(f"  leaf table + first CTA barrier (stamp 14): mean {(t2[:, 14] - t2[:, 0]).mean():8.0f}")
print(f"  GEMM body entered / mbarriers initialised (stamps 13, 15; single GPU only): {(t2[32:128, 13] - t2[32:128, 0]).mean():8.0f} {(t2[32:128, 15] - t2[32:128, 0]).mean():8.0f}")
gl = ["prologue done", "dependency wait passed", "first operands landed", "all MMAs issued", "accumulator complete (epilogue)", "tile staged in smem", "partial tile written"]
print("  GEMM body, cycles since kernel start (mean over GEMM CTAs 32..127):")
for k in range(7):
    print(f"    {gl[k]:34s} {(t2[32:128, 6 + k] - t2[32:128, 0]).mean():8.0f}")
print("  total per CTA: mean", (t2[:, 5] - t2[:, 0]).mean(), "max", (t2[:, 5] - t2[:, 0]).max())
