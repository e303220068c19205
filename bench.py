#!/usr/bin/env python
"""bench.py -- learner gradient-steps/sec of the D4PG hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # B200 arm (torchrun for N>1)
    python bench.py --impl reference --steps K --warmup W    # CPU arm: the reference's own DDPG.train (oracle/_ref)

Workload (config.workload = "c2"): |s|=17 |a|=6, 51 atoms, batch 256 per GPU, prioritized
replay capacity 2^20 per GPU (full), fp32-accurate arithmetic (3xTF32 on tcgen05, fp32 accumulate: the 1e-5
parity bar of the golden tests).  One step = everything DDPG.train() does (ddpg.py:200-255).  Weak scaling:
every rank owns a replay shard and a 256-row minibatch; the flat gradient is summed over the ranks once per
step (fused into the dW / Adam kernels over NVLink peer memory; NCCL all-reduce as fallback).  `value` counts
batch-256 gradient steps over all ranks per second (N x iterations/s).
"""
import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = {
    "c2": dict(obs=17, act=6, atoms=51, batch=256, cap=1 << 20, v_min=-50.0, v_max=0.0, n_steps=1, proj="reference"),
    "c3": dict(obs=376, act=17, atoms=51, batch=1024, cap=1000000, v_min=-50.0, v_max=0.0, n_steps=1, proj="reference"),
    "c5": dict(obs=17, act=6, atoms=101, batch=4096, cap=1 << 20, v_min=-150.0, v_max=150.0, n_steps=5, proj="nstep"),
}
H = 256
METRIC = "learner grad-steps/sec (batch 256, 51 atoms)"


def algorithmic(cfg):
    """SURVEY.md section 8d: FLOPs and bytes per gradient step."""
    S, A, N, B, cap = cfg["obs"], cfg["act"], cfg["atoms"], cfg["batch"], cfg["cap"]
    log2cap = int(np.ceil(np.log2(cap)))
    Pa = S * H + H + 2 * (H * H + H) + H * A + A
    Pc = S * H + H + (H + A) * H + H + H * H + H + H * N + N
    mac_a = S * H + 2 * H * H + H * A
    mac_c = S * H + (H + A) * H + H * H + H * N
    flops = 2 * B * (4 * mac_a + 6 * mac_c)
    gemm_bytes = (3 * Pa + 5 * Pc) * 4
    byts = (B * (2 * S + A + 2) * 4 + B * log2cap * 4 + B * (1 + log2cap) * 2 * 2 * 4 + 3 * B * N * 4
            + 7 * (Pa + Pc) * 4 + 3 * (Pa + Pc) * 4 + gemm_bytes)
    return dict(P=Pa + Pc, Pa=Pa, Pc=Pc, flops=flops, bytes=byts, gemm_bytes=gemm_bytes)


def config_dict(name, world):
    """The workload, identical in both arms (the driver compares them key by key)."""
    cfg = CFG[name]
    return {"workload": name, "batch_per_gpu": cfg["batch"], "global_batch": cfg["batch"] * world, "obs_dim": cfg["obs"],
            "act_dim": cfg["act"], "n_atoms": cfg["atoms"], "replay_capacity_per_gpu": cfg["cap"], "n_steps": cfg["n_steps"],
            "parallelism": "dp%d" % world}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tf=p.get("bf16_tflops_sustained", p.get("bf16_tflops")), src="measured")
    return dict(hbm=6650.0, tf=1590.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clock / throttle-reason samples during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(self.samples)}


def synth(cfg, n, seed):
    """SURVEY.md section 8d synthetic transitions (fp32-representable)."""
    rng = np.random.RandomState(seed)
    S, A = cfg["obs"], cfg["act"]
    return (rng.randn(n, S).astype(np.float32), rng.uniform(-1, 1, (n, A)).astype(np.float32),
            (-3.0 * rng.rand(n)).astype(np.float32).astype(np.float64), rng.randn(n, S).astype(np.float32),
            np.zeros(n, dtype=bool))


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's DDPG.train (the reference itself is Python and
# cannot travel to the GPU box; oracle/ is pinned bit-exact to it, see oracle/__init__.py)
# ------------------------------------------------------------------------------------------
def cpu_arm(cfg, steps, warmup, budget_s=25.0):
    import torch
    from oracle import d4pg_oracle as O
    info = {"type": "categorical", "v_min": cfg["v_min"], "v_max": cfg["v_max"], "n_atoms": cfg["atoms"]}
    B, cap = cfg["batch"], cfg["cap"]
    ncores = len(os.sched_getaffinity(0))
    best = None
    for threads in sorted({1, ncores}):
        torch.set_num_threads(threads)
        torch.manual_seed(0); random.seed(0)
        lo = O.LearnerOracle(cfg["obs"], cfg["act"], info, n_steps=cfg["n_steps"],
                             projection="live" if cfg["proj"] == "reference" else "nstep")
        ob = O.PrioritizedReplayOracle(cap, 0.6, cfg["obs"], cfg["act"])
        ob.add_batch(*synth(cfg, cap, 0))
        sched = O.LinearScheduleOracle(100000, 1.0, 0.4)

        def one():
            us = [random.random() for _ in range(B)]
            batch = ob.sample(B, sched.value(), us)
            out = lo.train_step(*batch[:5])
            ob.update_priorities(batch[6], out["prio"])
        for _ in range(warmup):
            one()
        t0 = time.perf_counter()
        done = 0
        while done < steps and (time.perf_counter() - t0) < budget_s / 2:
            one()
            done += 1
        dt = time.perf_counter() - t0
        rate = done / dt
        if best is None or rate > best["value"]:
            best = dict(value=rate, cores=threads, done=done, dt=dt)
    return best


def cpu_arm_reference(cfg, steps, warmup, budget_s=25.0, n_fill=1 << 17):
    """The UNMODIFIED reference (oracle/_ref = its modules byte-compiled by oracle/build_ref.py, or /root/reference where
    that exists) behind the 4-item compat shim, wired as main.py:382-392 wires it, driven through its public API only:
    PrioritizedReplayBuffer.add() x n_fill, then DDPG.train(global).  The buffer has the workload's capacity (tree depth
    20 for 2^20) but is filled with `n_fill` transitions: a million Python add() calls would not fit the time budget."""
    import torch
    from oracle import ref_shim
    info = {"type": "categorical", "v_min": cfg["v_min"], "v_max": cfg["v_max"], "n_atoms": cfg["atoms"]}
    B, cap = cfg["batch"], cfg["cap"]
    ncores = len(os.sched_getaffinity(0))
    n_fill = min(n_fill, cap)
    S, A, R, S2, D = synth(cfg, n_fill, 0)
    best = None
    for threads in sorted({1, ncores}):
        torch.set_num_threads(threads)
        g, l, oa, oc = ref_shim.make_learner_pair(cfg["obs"], cfg["act"], info, B, cap, prioritized_replay=True,
                                                  n_steps=cfg["n_steps"], seed=0)
        for i in range(n_fill):
            l.replayBuffer.add(S[i], A[i], float(R[i]), S2[i], bool(D[i]))
        for _ in range(warmup):
            l.train(g)
        t0 = time.perf_counter()
        done = 0
        while done < steps and (time.perf_counter() - t0) < budget_s / 2:
            l.train(g)
            done += 1
        dt = time.perf_counter() - t0
        rate = done / dt
        if best is None or rate > best["value"]:
            best = dict(value=rate, cores=threads, done=done, dt=dt)
        del g, l, oa, oc
    best["n_fill"] = n_fill
    return best


def cpu_baseline(cfg, name, steps, warmup, budget_s):
    """cpu_baseline object of the JSON line: the reference itself when oracle/_ref travelled, else the oracle port."""
    from oracle import ref_shim
    ncores = len(os.sched_getaffinity(0))
    if ref_shim.available():
        r = cpu_arm_reference(cfg, steps, warmup, budget_s)
        return r, {"value": r["value"], "unit": "steps/s", "cores": r["cores"], "kind": "reference",
                   "sample": "%d DDPG.train() calls of the UNMODIFIED reference (ddpg.py:200-255 + prioritized_replay_memory.py, "
                             "%s) on workload %s: PER capacity %d (tree depth %d), %d transitions added through add(); host has %d "
                             "cores, best of torch threads {1,%d} = %d" % (
                                 r["done"], "from /root/reference" if ref_shim.source_available() else "oracle/_ref, byte-compiled from /root/reference",
                                 name, cfg["cap"], int(np.ceil(np.log2(cfg["cap"]))), r["n_fill"], ncores, ncores, r["cores"])}
    r = cpu_arm(cfg, steps, warmup, budget_s)
    return r, {"value": r["value"], "unit": "steps/s", "cores": r["cores"], "kind": "port",
               "sample": "%d steps of the oracle port (restatement of ddpg.py:200-255 + PER, pinned bit-for-bit to the reference; "
                         "oracle/_ref was not present), workload %s, buffer full; host has %d cores, best of torch threads {1,%d} = %d" % (
                             r["done"], name, ncores, ncores, r["cores"])}


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CFG[args.config]
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    r, cpu = cpu_baseline(cfg, args.config, args.steps, max(args.warmup, 3), 50.0)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "steps_timed": r["done"], "warmup": args.warmup, "ms_per_step": 1e3 / r["value"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args.config, world),
            "cpu_baseline": cpu,
            "e2e": {"value": r["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def dump_outputs(dd, out_dir):
    """What a caller of the timed path receives after its last step, as DIR/<name>.npy: the losses, the sampled
    batch (indices, IS weights, TD errors, new priorities) and every parameter of the four networks."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"losses": np.array(dd.last_losses(), dtype=np.float32)}
    for k, v in dd.last_batch_info().items():
        out["batch_" + k] = v.cpu().numpy().astype(np.float64 if k == "idx" else np.float32)
    for net in ("actor", "critic", "actor_target", "critic_target"):
        for k, v in getattr(dd, net).state_dict().items():
            out["%s.%s" % (net, k)] = v.cpu().numpy().astype(np.float32)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def gpu_main(args):
    import torch
    import d4pg_b200 as d4pg
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    comm = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        comm = d4pg.dist.Comm()
    cfg = CFG[args.config]
    info = {"type": "categorical", "v_min": cfg["v_min"], "v_max": cfg["v_max"], "n_atoms": cfg["atoms"]}
    B, cap = cfg["batch"], cfg["cap"]

    def make(sampling):
        torch.manual_seed(0); random.seed(0)            # identical replicas on every rank
        dd = d4pg.DDPG(cfg["obs"], cfg["act"], memory_size=cap, batch_size=B, critic_dist_info=info,
                       n_steps=cfg["n_steps"], projection=cfg["proj"], sampling=sampling, philox_seed=1234 + rank,
                       comm=comm, precision=args.precision, chain={0: "levels", 1: "cluster"}[args.chain])
        dd.assign_global_optimizer(d4pg.SharedAdam(dd.actor.parameters(), lr=1e-3),
                                   d4pg.SharedAdam(dd.critic.parameters(), lr=1e-3))
        dd.replayBuffer.add_batch(*synth(cfg, cap, seed=rank))     # this rank's shard, resident in HBM
        return dd

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- value: inputs resident in HBM, device-side sampling, CUDA-graph replay -------------
    dd = make("device")
    # untimed warm-up: at least W steps, issued so that every CUDA-graph variant of the step (cold / warm, both halves of
    # the double-buffered batch, the 4-step replay graphs) is captured and instantiated before the timed region
    capture_steps = 0
    for n in (1, 4, 1, 4, 1):
        dd.train_n(n); capture_steps += n
    dd.train_n(max(args.warmup, 3))                 # the W requested warm-up steps
    stream = dd._learner.stream
    sampler = ClockSampler(local)
    sampler.start()
    # the timed region = EXACTLY K steps between barrier + synchronize on both sides, CUDA events on the learner stream,
    # max over ranks; --steps K is the number of timed steps.  A short region (K = 20 steps lasts ~2 ms) can be measured
    # R = --repeats times back to back, and the MEDIAN region is reported (every region is listed)
    regions = []
    for _ in range(max(1, args.repeats)):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
        dd.train_n(args.steps)                      # K graph replays, no host work in between
        with torch.cuda.stream(stream):
            e1.record(stream)
        barrier()
        regions.append(max_over_ranks(e0.elapsed_time(e1)))
    if args.dump_outputs and rank == 0:
        dump_outputs(dd, args.dump_outputs)
    ms = float(np.median(regions))
    kernels = dd.kernels_per_step()
    exchange = comm.exchange_mode() if comm is not None else "single"
    lc, la = dd.last_losses()
    assert np.isfinite(lc) and np.isfinite(la)
    ms_per_step = ms / args.steps
    value = world * 1e3 / ms_per_step
    # data-parallel replicas must stay bit-identical: hash actor || critic || both targets on every rank and compare
    replicas_identical = None
    if world > 1:
        import torch.distributed as dist
        flat = torch.cat([dd.actor.flat_params(), dd.critic.flat_params(), dd.actor_target.flat_params(),
                          dd.critic_target.flat_params()]).view(torch.int32).to(torch.int64)
        w = torch.arange(1, flat.numel() + 1, device=flat.device, dtype=torch.int64) * 2654435761
        h = torch.stack([(flat * w).sum(), flat.sum()])                   # 2 x 64-bit (wrapping) checksums
        hs = [torch.zeros_like(h) for _ in range(world)]
        dist.all_gather(hs, h)
        replicas_identical = bool(all(torch.equal(hs[0], x) for x in hs))
        assert replicas_identical, "data-parallel replicas diverged"

    # ---- per-launch device times (eager step, CUDA events on the launching stream) -----------
    prof = {}
    for _ in range(5):
        seen = {}
        for name, t in dd.profile_step():
            k = seen.get(name, 0); seen[name] = k + 1
            prof.setdefault("%s#%d" % (name, k), []).append(t)
    alg = algorithmic(cfg)
    pk = peaks()
    S_, A_d, N_, Pa, Pc = cfg["obs"], cfg["act"], cfg["atoms"], alg["Pa"], alg["Pc"]
    # algorithmic bytes of one launch of each MLP kernel class (DESIGN.md section 2): weights read once,
    # batch inputs once, gradients written once
    kinds = {}
    if any(k.startswith("launch_mlp_tc_chain") for k in prof):
        kinds["launch_mlp_tc_chain#0"] = ("mlp_tc_chain_kernel (3 forward chains, 20 layers, 1 launch)", 4 * (2 * Pa + 3 * Pc) + 4 * B * (2 * S_ + A_d), "fwd")
        kinds["launch_mlp_tc_chain#1"] = ("mlp_tc_chain_kernel (2 dX chains, 9 layers, 1 launch)", 4 * (Pa + 2 * Pc) + 8 * B * N_, "bwd")
        kinds["gemm_wide_launch#0"] = ("gemm_wide_kernel (9 dW problems, 1 launch)", 4 * (Pa + Pc) + 4 * B * 9 * H, "dw")
    elif any(k.startswith("launch_mlp_chain") for k in prof):
        kinds["launch_mlp_chain#0"] = ("mlp_chain_kernel (3 forward chains, 20 layers, 1 launch)", 4 * (2 * Pa + 3 * Pc) + 4 * B * (2 * S_ + A_d), "fwd")
        kinds["launch_mlp_chain#1"] = ("mlp_chain_kernel (2 dX chains, 9 layers, 1 launch)", 4 * (Pa + 2 * Pc) + 8 * B * N_, "bwd")
        kinds["gemm_wide_launch#0"] = ("gemm_wide_kernel (9 dW problems, 1 launch)", 4 * (Pa + Pc) + 4 * B * 9 * H, "dw")
    else:
        n_gemm = len([k for k in prof if k.startswith("gemm_launch")])
        for k in prof:
            if k.startswith("gemm_launch"):
                kinds[k] = ("%s (MLP level, %d launches/step)" % ("gemm_ffma_kernel" if args.precision == "fp32" else "gemm_tc2_kernel", n_gemm),
                            alg["gemm_bytes"] / max(n_gemm, 1), "level")
    roofline = None
    if kinds:
        mlp_ms = {k: float(np.mean(prof[k])) for k in kinds if k in prof}
        if "launch_mlp_chain#0" in mlp_ms or "launch_mlp_tc_chain#0" in mlp_ms:
            top = max(mlp_ms, key=mlp_ms.get)
            name, nbytes, _ = kinds[top]
            t_ms = mlp_ms[top]
            flops = alg["flops"] * {"fwd": 0.5, "bwd": 0.25, "dw": 0.25}[kinds[top][2]]
        else:                                   # all levels are one kernel class: average launch
            top = sorted(mlp_ms)[0]
            name, nbytes, _ = kinds[top]
            t_ms = float(np.mean(list(mlp_ms.values())))
            flops = alg["flops"] / len(mlp_ms)
        ach = nbytes / (t_ms * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(name.split(" ")[0] + ":" + kinds[top][2])
        # the MLP layers are dense contractions: the roof that bounds them is the tensor pipe (SURVEY.md section 8d);
        # `achieved` = algorithmic FLOPs of the launch (2*M*N*K of its layers, the fp32 math -- the 3xTF32 split issues 3x
        # as many tensor-core MACs at the TF32 rate, half the bf16 rate) / its CUDA-event duration; the HBM view is kept
        tf = flops / (t_ms * 1e-3) / 1e12
        roofline = {"kernel": name, "bound": "tensor", "achieved": tf, "peak": pk["tf"], "unit": "TFLOP/s",
                    "frac": tf / pk["tf"], "traffic": traffic,
                    "peak_source": pk["src"] + " (sustained dense bf16 cuBLAS; no TF32 figure is measured on this pool, nominal TF32 = bf16 / 2)",
                    "avg_launch_us": t_ms * 1e3, "algorithmic_flops_per_launch": int(flops),
                    "algorithmic_bytes_per_launch": int(nbytes),
                    "hbm": {"achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"]}}
    step_roof = {"hbm_frac": alg["bytes"] / (ms_per_step * 1e-3) / 1e9 / pk["hbm"],
                 "tensor_frac": alg["flops"] / (ms_per_step * 1e-3) / 1e12 / pk["tf"],
                 "algorithmic_bytes": alg["bytes"], "algorithmic_flops": alg["flops"]}
    launch_breakdown = {k: round(float(np.mean(v)) * 1e3, 2) for k, v in prof.items()}   # us per launch
    del dd

    # ---- e2e: public API with host buffers: per step H2D of new transitions + uniforms, D2H loss
    dd = make("reference")
    n_new = B
    S, A_, R, S2, D = synth(cfg, n_new * 8, seed=100 + rank)
    pin = [torch.from_numpy(x).pin_memory() for x in (S, A_, R, S2, D)]
    h2d = B * 8 + n_new * ((2 * cfg["obs"] + cfg["act"]) * 4 + 8 + 1)
    d2h = 16

    def e2e_step(i, first=False):
        lo = (i % 8) * n_new
        dd.replayBuffer.add_batch(*[p[lo:lo + n_new] for p in pin])      # H2D from pinned host memory
        dd.train()                                                        # host MT19937 uniforms -> H2D; queues the D2H of its losses
        # every step's result is read on the host, one step late: the read of step k-1 overlaps step k on the GPU
        # (the last step's own result is read before the clock stops, below)
        return None if first else dd.last_losses(lag=1)
    for i in range(max(args.warmup, 3)):
        e2e_step(i, first=(i == 0))
    dd.last_losses()
    barrier()
    t0 = time.perf_counter()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    e2e_steps = args.steps * max(1, args.repeats)      # same number of steps as the device-timed regions together
    for i in range(e2e_steps):
        e2e_step(i)
    lc_e, la_e = dd.last_losses()                   # D2H result of the final step, inside the timed region
    assert np.isfinite(lc_e) and np.isfinite(la_e)
    ev1.record()
    barrier()
    e2e_ms = max_over_ranks(max(ev0.elapsed_time(ev1), (time.perf_counter() - t0) * 1e3))
    e2e_value = world * e2e_steps / (e2e_ms * 1e-3)
    sampler.stop_flag = True                        # clocks were sampled through both timed regions
    del dd

    # ---- CPU baseline beside it (rank 0, N=1 only) ---------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        _, cpu = cpu_baseline(cfg, args.config, 200, 3, 24.0)
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict(args.config, world),
                "timing": {"regions_ms": [round(x, 4) for x in regions], "reported": "median region", "steps_per_region": args.steps,
                           "graph_capture_steps_before_warmup": capture_steps, "warmup_steps": max(args.warmup, 3)},
                "replicas_identical": replicas_identical,
                "implementation": {"step_plan": "levels (one launch per dependency level; the library's plan above 512 rows)" if (B > 512 or not args.chain) else "cluster chains",
                           "gradient_exchange": exchange,
                           "precision": {"fp32": "exact fp32 FFMA tiles", "tf32x3": "3xTF32 on tcgen05 tensor cores (hi/lo split, fp32 accumulate in TMEM; meets the 1e-5 parity bar)", "tf32": "one TF32 tcgen05 pass (not parity-grade)"}[args.precision],
                           "l2": "inputs larger than L2: replay store %.0f MB + trees %.0f MB per GPU, rows sampled at "
                                 "random; parameters (%.1f MB) are L2-resident by design" % (
                                     cap * ((2 * cfg["obs"] + cfg["act"]) * 4 + 9) / 1e6, 16 * cap / 1e6 * 1.05, alg["P"] * 16 / 1e6)},
                "clocks": sampler.summary(), "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": h2d,
                                                     "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps,
                                                     "how": "per step: add_batch of 256 new transitions from pinned host memory (H2D), train() with host-drawn "
                                                            "MT19937 uniforms (H2D), its losses copied D2H; the host reads step k-1's losses while step k runs "
                                                            "(DDPG.last_losses(lag=1)), the final step's before the clock stops.  Host pipeline: add(k) and "
                                                            "sample(k) run on the learner's ingest stream behind step k-1's priority write-back, overlapping its "
                                                            "backward pass / dW / Adam (tree order update(k-1) -> add(k) -> sample(k) as in the reference)"},
                "gpu_launches": kernels * args.steps, "kernels_per_step": kernels,
                "roofline": roofline, "roofline_step": step_roof, "launch_us_per_step": launch_breakdown,
                "cpu_baseline": cpu, "losses": [lc, la]}
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CFG))
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--repeats", type=int, default=1, help="timed regions of K steps each; the median region is reported")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's outputs as DIR/<name>.npy")
    ap.add_argument("--precision", default="tf32x3", choices=["fp32", "tf32x3", "tf32"])
    ap.add_argument("--chain", type=int, default=1, help="MLP step plan: 1 = cluster-fused chains, 0 = one launch per level")
    args = ap.parse_args()
    if args.impl == "reference":
        reference_main(args)
    else:
        gpu_main(args)


if __name__ == "__main__":
    main()
