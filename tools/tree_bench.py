"""python tools/tree_bench.py : device time of one update_priorities call (256 leaves, capacity 2^20), CUDA events,
with an L2 flush between calls.  At this size the update runs the fast multi-CTA kernel (tree_update_fast_kernel)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import d4pg_b200 as d4pg
n, S, A, B = 1 << 20, 17, 6, 256
buf = d4pg.PrioritizedReplayBuffer(n, 0.6, obs_dim=S, act_dim=A, device="cuda")
rng = np.random.RandomState(0)
buf.add_batch(rng.randn(n, S).astype(np.float32), rng.uniform(-1, 1, (n, A)).astype(np.float32), -rng.rand(n), rng.randn(n, S).astype(np.float32), np.zeros(n, bool))
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
ts = []
for it in range(12):
    idx = torch.from_numpy(rng.randint(0, n, B).astype(np.int32)).cuda()
    pr = torch.from_numpy(rng.rand(B).astype(np.float32) + 1e-6).cuda()
    if it % 2: flush.zero_()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); buf.update_priorities(idx, pr); e1.record(); torch.cuda.synchronize()
    ts.append((it % 2, e0.elapsed_time(e1) * 1e3))
print("warm L2: %s us" % ["%.1f" % t for f, t in ts[2:] if not f])
print("flushed L2: %s us" % ["%.1f" % t for f, t in ts[2:] if f])
