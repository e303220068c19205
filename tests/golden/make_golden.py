#!/usr/bin/env python
"""Generate tests/golden/*.npz by RUNNING THE UNMODIFIED REFERENCE (/root/reference)
behind oracle/ref_shim.py.  Only runs in the build container; the fixtures it
writes are committed and travel to the GPU box.

    python tests/golden/make_golden.py

Generated with: Python 3.12.3, numpy 2.3.5 (NEP-50 dtype rules -> fp32 trees),
torch 2.11.0 CPU.  Re-running under other NumPy majors changes dtype semantics
(SURVEY.md H11).
"""
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_shim  # noqa: E402
from tests.helpers import NAMES, ScriptedEnv, digest, regen_init, transitions  # noqa: E402

INFO51 = {"type": "categorical", "v_min": -50.0, "v_max": 0.0, "n_atoms": 51}
INFO101 = {"type": "categorical", "v_min": -150.0, "v_max": 150.0, "n_atoms": 101}
INFO_PEND = {"type": "categorical", "v_min": -300.0, "v_max": 0.0, "n_atoms": 51}


def softmax_rows(rng, B, N, sharp=1.0):
    z = (rng.randn(B, N) * sharp).astype(np.float32)
    return torch.softmax(torch.from_numpy(z), dim=1).numpy()


def ref_project(ref, info, gamma, n_steps, probs, r, done, live=True):
    B = probs.shape[0]
    d = ref.ddpg.DDPG(3, 1, batch_size=B, gamma=gamma, critic_dist_info=info,
                      prioritized_replay=False, n_steps=n_steps, memory_size=8)
    if live:
        return d.reproject2(probs, r, done)
    return d.reproj_categorical_dist(probs.astype(np.float64), r, done.astype(np.float64))


def gen_projection(ref):
    rng = np.random.RandomState(1234)
    out = {}
    # KATs from SURVEY.md section 8c(1)
    p = softmax_rows(rng, 4, 51)
    r = np.array([-1.0, -1.0, -60.0, 5.0])
    done = np.zeros(4, dtype=bool)
    out["kat_nt_probs"], out["kat_nt_r"], out["kat_nt_done"] = p, r, done
    out["kat_nt_m"] = ref_project(ref, INFO51, 0.99, 1, p, r, done)
    r = np.array([-1.6346495489906907, -0.3, -49.99, -33.3])
    done = np.ones(4, dtype=bool)
    out["kat_t_probs"], out["kat_t_r"], out["kat_t_done"] = p, r, done
    out["kat_t_m"] = ref_project(ref, INFO51, 0.99, 1, p, r, done)
    r = np.array([-1.0, 0.0, -50.0, -77.0])          # last one clamps to bin 0
    out["kat_ti_probs"], out["kat_ti_r"], out["kat_ti_done"] = p, r, done
    out["kat_ti_m"] = ref_project(ref, INFO51, 0.99, 1, p, r, done)

    # random batches: continuous / integer (HER-style) rewards, 0 % / 5 % / 100 % terminal;
    # terminal rows never mix integer and non-integer b_j (SURVEY.md H6)
    case = 0
    for info, B in ((INFO51, 256), (INFO101, 192), (INFO_PEND, 64)):
        N = info["n_atoms"]
        for rew_kind in ("cont", "int"):
            for term in (0.0, 0.05, 1.0):
                p = softmax_rows(rng, B, N, sharp=2.0)
                if rew_kind == "cont":
                    r = (-3.0 * rng.rand(B)).astype(np.float32).astype(np.float64)
                    if info is INFO101:
                        r = (200.0 * (rng.rand(B) - 0.5)).astype(np.float32).astype(np.float64)
                else:
                    # HER-style {0,-1} rewards scaled to the atom spacing so every
                    # terminal b_j is an integer (all-eq terminal batch, no H6 crash)
                    dl = (info["v_max"] - info["v_min"]) / (N - 1)
                    r = -dl * rng.randint(0, 2, size=B).astype(np.float64)
                done = rng.rand(B) < term
                k = "rand%d" % case
                out[k + "_meta"] = np.array([info["v_min"], info["v_max"], N, 0.99])
                out[k + "_probs"], out[k + "_r"], out[k + "_done"] = p, r, done
                out[k + "_m"] = ref_project(ref, info, 0.99, 1, p, r, done)
                case += 1
    out["n_rand"] = np.array(case)

    # n-step (config 5): reproj_categorical_dist at n_steps=5, 101 atoms
    for i, term in enumerate((0.0, 0.05)):
        B = 128
        p = softmax_rows(rng, B, 101, sharp=2.0)
        r = (40.0 * (rng.rand(B) - 0.5)).astype(np.float32).astype(np.float64)
        r[:8] = np.array([0., 3., -3., 150., -150., 149.999, 6., -9.])   # integer b_j hits
        done = rng.rand(B) < term
        k = "nstep%d" % i
        out[k + "_probs"], out[k + "_r"], out[k + "_done"] = p, r, done
        out[k + "_m"] = ref_project(ref, INFO101, 0.99, 5, p, r, done, live=False)
    np.savez_compressed(os.path.join(HERE, "projection.npz"), **out)
    print("projection.npz:", len(out), "arrays")


def dump_tree(buf):
    s = np.array([float(x) for x in buf._it_sum._value], dtype=np.float64)
    m = np.array([float(x) for x in buf._it_min._value], dtype=np.float64)
    return s, m


def gen_tree(ref):
    """prioritized_replay_memory.py state after fill + K rounds of update_priorities
    (f32 priorities, duplicate indices), plus sample() indices / weights."""
    out = {}
    rng = np.random.RandomState(77)
    for name, size, n_fill in (("full", 1000, 1000), ("part", 3000, 1733), ("wrap", 256, 700)):
        buf = ref.prioritized_replay_memory.PrioritizedReplayBuffer(size, alpha=0.6)
        for i in range(n_fill):
            buf.add(np.full(2, i, np.float32), np.zeros(1, np.float32), -1.0, np.zeros(2, np.float32), False)
        B = 64
        rounds = 5
        out[name + "_meta"] = np.array([size, n_fill, B, rounds])
        random.seed(4242)
        us, idxs, ws, betas = [], [], [], []
        upd_i, upd_p = [], []
        s0, m0 = dump_tree(buf)
        out[name + "_sum_r0"], out[name + "_min_r0"] = s0, m0
        for k in range(rounds):
            st = random.getstate()
            u = np.array([random.random() for _ in range(B)])
            random.setstate(st)
            beta = 0.4 + 0.1 * k
            samp = buf.sample(B, beta)
            us.append(u)
            idxs.append(np.array(samp[6], dtype=np.int64))
            ws.append(np.array(samp[5], dtype=np.float64))
            betas.append(beta)
            # priorities as the learner produces them: f32 ndarray in (0, 1+1e-6]
            ii = np.array(samp[6], dtype=np.int64)
            if k % 2 == 1:
                ii[1::4] = ii[0::4]                      # force duplicate indices
            pr = (np.abs(rng.rand(B).astype(np.float32)) + np.float32(1e-6)).astype(np.float32)
            if k == 3:
                pr[5] = np.float32(1.000001)             # raises max_priority to an f32 value
            buf.update_priorities(list(ii), pr)
            upd_i.append(ii)
            upd_p.append(pr)
            s, m = dump_tree(buf)
            out["%s_sum_r%d" % (name, k + 1)] = s
            out["%s_min_r%d" % (name, k + 1)] = m
            if k == 3:                                   # adds after max_priority became f32
                for j in range(7):
                    buf.add(np.zeros(2, np.float32), np.zeros(1, np.float32), -1.0, np.zeros(2, np.float32), False)
                s, m = dump_tree(buf)
                out[name + "_sum_after_add"], out[name + "_min_after_add"] = s, m
        out[name + "_u"] = np.stack(us)
        out[name + "_idx"] = np.stack(idxs)
        out[name + "_w"] = np.stack(ws)
        out[name + "_beta"] = np.array(betas)
        out[name + "_upd_idx"] = np.stack(upd_i)
        out[name + "_upd_prio"] = np.stack(upd_p)
        out[name + "_max_priority"] = np.array(float(buf._max_priority))
    np.savez_compressed(os.path.join(HERE, "tree.npz"), **out)
    print("tree.npz:", len(out), "arrays")


def sd_np(module):
    return {k: v.detach().clone().numpy() for k, v in module.state_dict().items()}


STRIDE = 31


def compact(out, key, arr):
    """Big tensors are stored as a strided subsample + f64 checksums (keeps the
    fixtures small); tensors <= 4096 elements are stored whole."""
    arr = np.asarray(arr)
    if arr.size <= 4096:
        out[key] = arr
    else:
        flat = arr.reshape(-1)
        out[key + "__sub"] = flat[::STRIDE].copy()
        out[key + "__chk"] = np.array([flat.astype(np.float64).sum(),
                                       np.abs(flat.astype(np.float64)).sum(), flat.size])


def train_data(seed, n_fill, obs_dim, act_dim, term_p):
    """The transitions of a train_*.npz fixture (also used by the tests to REGENERATE them when a fixture stores
    only the seed: numpy's RandomState streams are stable across versions)."""
    rng = np.random.RandomState(seed + 1)
    S = rng.randn(n_fill, obs_dim).astype(np.float32)
    A = rng.uniform(-1, 1, (n_fill, act_dim)).astype(np.float32)
    R = (-3.0 * rng.rand(n_fill)).astype(np.float32).astype(np.float64)
    S2 = rng.randn(n_fill, obs_dim).astype(np.float32)
    # terminal rows get non-integer rewards only (no H6 mixing)
    D = rng.rand(n_fill) < term_p
    return S, A, R, S2, D


def gen_train(ref, tag, obs_dim, act_dim, info, B, mem, n_fill, per, steps, term_p, seed, n_steps=1, store_data=True):
    """`steps` consecutive DDPG.train() calls (ddpg.py:200-255) from a saved state."""
    out = {}
    g, l, oa, oc = ref_shim.make_learner_pair(obs_dim, act_dim, info, B, mem,
                                              prioritized_replay=per, seed=seed, n_steps=n_steps)
    S, A, R, S2, D = train_data(seed, n_fill, obs_dim, act_dim, term_p)
    for i in range(n_fill):
        l.replayBuffer.add(S[i], A[i], float(R[i]), S2[i], bool(D[i]))
    out["meta"] = np.array([obs_dim, act_dim, info["n_atoms"], B, mem, n_fill, int(per), steps])
    out["dist"] = np.array([info["v_min"], info["v_max"]])
    out["n_steps"] = np.array(n_steps)
    if store_data:
        out["S"], out["A"], out["R"], out["S2"], out["D"] = S, A, R, S2, D
    else:                                   # big fixtures: the tests regenerate the transitions from the seed
        out["term_p"] = np.array(term_p)
        compact(out, "S", S); compact(out, "R", R)
    # initial weights are re-creatable from `seed` (oracle.init_actor/init_critic consume
    # the RNG exactly like models.py); the subsample pins them
    out["seed"] = np.array(seed)
    for net, mod in (("actor", l.actor), ("critic", l.critic)):
        for k, v in sd_np(mod).items():
            compact(out, "init_%s_%s" % (net, k), v)

    rec = {}
    orig_reproj = l.reproject2

    def reproj(tz, r, d):
        m = orig_reproj(tz, r, d)
        rec["tz"], rec["m"] = np.array(tz), np.array(m)
        return m
    l.reproject2 = reproj
    orig_cf = l.critic.forward
    qs = []

    def cf(s, a):
        q = orig_cf(s, a)
        qs.append(q.detach().clone().numpy())
        return q
    l.critic.forward = cf
    orig_oc, orig_oa = oc.step, oa.step

    def oc_step():
        rec["g_critic"] = [p.grad.detach().clone().numpy() for p in g.critic.parameters()]
        return orig_oc()

    def oa_step():
        rec["g_actor"] = [p.grad.detach().clone().numpy() for p in g.actor.parameters()]
        return orig_oa()
    oc.step, oa.step = oc_step, oa_step
    if per:
        orig_up = l.replayBuffer.update_priorities

        def up(idx, pr):
            rec["idx"], rec["prio"] = np.array(idx, dtype=np.int64), np.array(pr)
            return orig_up(idx, pr)
        l.replayBuffer.update_priorities = up

    names = [k for k, _ in l.critic.named_parameters()]
    for t in range(steps):
        random.seed(9000 + t)
        st = random.getstate()
        if per:
            out["u_%d" % t] = np.array([random.random() for _ in range(B)])
        else:
            pos = random.sample(range(len(l.replayBuffer.buffer)), B)
            out["idx_%d" % t] = np.array(pos, dtype=np.int64)
        random.setstate(st)
        del qs[:]
        l.train(g)
        m, q = torch.from_numpy(rec["m"]), torch.from_numpy(qs[0])
        out["loss_critic_%d" % t] = (-(m * torch.log(q + 1e-10)).sum(dim=1).mean()).numpy()   # ddpg.py:217
        z = torch.from_numpy(l.bin_centers).float()
        out["loss_actor_%d" % t] = (-torch.from_numpy(qs[1]).matmul(z).mean()).numpy()       # ddpg.py:238
        for key, arr in (("target_probs_%d" % t, rec["tz"]), ("m_%d" % t, rec["m"]), ("q_%d" % t, qs[0]), ("q_pi_%d" % t, qs[1])):
            if store_data:
                out[key] = arr
            else:
                compact(out, key, arr)
        if per:
            out["idx_%d" % t], out["prio_%d" % t] = rec["idx"], rec["prio"]
            s, mn = dump_tree(l.replayBuffer)
            out["tree_sum_%d" % t], out["tree_min_%d" % t] = s, mn
        for nme, garr in zip(names, rec["g_critic"]):
            compact(out, "g_critic_%s_%d" % (nme, t), garr)
        for nme, garr in zip(names, rec["g_actor"]):
            compact(out, "g_actor_%s_%d" % (nme, t), garr)
        for net, mod in (("actor", l.actor), ("critic", l.critic)):
            for k, v in sd_np(mod).items():
                compact(out, "%s_%s_%d" % (net, k, t), v)
        if t == steps - 1:
            for net, mod in (("actor_target", l.actor_target), ("critic_target", l.critic_target)):
                for k, v in sd_np(mod).items():
                    compact(out, "%s_%s_%d" % (net, k, t), v)
            for net, opt, mod in (("actor", oa, g.actor), ("critic", oc, g.critic)):
                for (k, _), p in zip(mod.named_parameters(), mod.parameters()):
                    compact(out, "adam_m_%s_%s_%d" % (net, k, t), opt.state[p]["exp_avg"].clone().numpy())
                    compact(out, "adam_v_%s_%s_%d" % (net, k, t), opt.state[p]["exp_avg_sq"].clone().numpy())
    np.savez_compressed(os.path.join(HERE, "train_%s.npz" % tag), **out)
    print("train_%s.npz:" % tag, len(out), "arrays")


def gen_init(ref):
    """Seeded weight init of models.py:16-30,52-73 (RNG-consumption parity)."""
    out = {}
    torch.manual_seed(5)
    a = ref.models.actor(17, 6)
    c = ref.models.critic(17, 6, INFO51)
    for k, v in sd_np(a).items():
        compact(out, "actor_" + k, v)
    for k, v in sd_np(c).items():
        compact(out, "critic_" + k, v)
    x = torch.randn(5, 17)
    act = torch.rand(5, 6) * 2 - 1
    out["x"], out["act"] = x.numpy(), act.numpy()
    out["actor_out"] = a(x).detach().numpy()
    out["critic_out"] = c(x, act).detach().numpy()
    np.savez_compressed(os.path.join(HERE, "init.npz"), **out)
    print("init.npz:", len(out), "arrays")


def gen_nstep(ref):
    """Replay.initialize (replay_memory.py:21-59): n-step return accumulation at insert, n_steps=5."""
    out = {}
    env = ScriptedEnv()
    np.random.seed(321)
    rp = ref.replay_memory.Replay(64, env, n_steps=5, gamma=0.99)
    rp.initialize(init_length=40)
    out["meta"] = np.array([5, 40, len(rp.buffer), len(env.log)])
    out["gamma"] = np.array(0.99)
    out["buf_s"] = np.stack([np.asarray(b[0], dtype=np.float64).reshape(-1) for b in rp.buffer])
    out["buf_a"] = np.stack([np.asarray(b[1], dtype=np.float64) for b in rp.buffer])
    out["buf_r"] = np.array([b[2] for b in rp.buffer], dtype=np.float64)
    out["buf_s2"] = np.stack([np.asarray(b[3], dtype=np.float64) for b in rp.buffer])
    out["buf_d"] = np.array([bool(b[4]) for b in rp.buffer])
    for i, e in enumerate(env.log):
        for k in ("s", "a", "r", "s2", "d"):
            out["ep%d_%s" % (i, k)] = np.asarray(e[k])
    np.savez_compressed(os.path.join(HERE, "nstep_init.npz"), **out)
    print("nstep_init.npz:", len(out), "arrays,", len(rp.buffer), "transitions from", len(env.log), "episodes")


def gen_baseline_sizes(ref):
    """Fixtures at the BASELINE.json sizes (VERDICT r1 item 6): c2 as configured (B=256), config-3 shapes
    (|s|=376, |a|=17, B=1024, small capacity), config-5 shapes (101 atoms, n_steps=5; train() at B=256 -- the live
    projection is reproject2 with gamma, SURVEY.md H5) and the n-step projection at B=4096."""
    gen_train(ref, "per_c2_b256", 17, 6, INFO51, 256, 2048, 2048, True, 3, 0.05, seed=21, store_data=False)
    gen_train(ref, "per_c3_b1024", 376, 17, INFO51, 1024, 2048, 2048, True, 2, 0.05, seed=22, store_data=False)
    gen_train(ref, "per_c5_b256", 17, 6, INFO101, 256, 2048, 2048, True, 2, 0.05, seed=23, n_steps=5, store_data=False)
    rng = np.random.RandomState(4096)
    B = 4096
    p = softmax_rows(rng, B, 101, sharp=2.0)
    r = (40.0 * (rng.rand(B) - 0.5)).astype(np.float32).astype(np.float64)
    done = rng.rand(B) < 0.05
    out = {"seed": np.array(4096), "B": np.array(B)}
    compact(out, "probs", p); compact(out, "r", r)
    out["done_count"] = np.array(int(done.sum()))
    compact(out, "m", ref_project(ref, INFO101, 0.99, 5, p, r, done, live=False))
    np.savez_compressed(os.path.join(HERE, "projection_c5_b4096.npz"), **out)
    print("projection_c5_b4096.npz:", len(out), "arrays")


def gen_oracle_vs_reference(ref):
    """What tests/test_oracle_vs_reference.py compares the oracle with: reproject2 on random batches, reproject2 vs
    reproj_categorical_dist at n_steps=5 (SURVEY H5), five DDPG.train() steps from a 650-transition PER buffer, and
    the indices _sample_proportional draws from a pristine 2^16 tree.  Inputs the test can regenerate exactly (seeded
    random.random() draws, the transitions) are pinned by their SHA-256; the softmax inputs are stored, since torch's
    CPU softmax rounds differently with the vector width.  Outputs are stored whole where small, else as SHA-256."""
    out = {}
    rng = np.random.RandomState(5)
    proj = {"probs": [], "r": [], "done": [], "m": []}
    for trial in range(6):
        B = 97
        d = ref.ddpg.DDPG(3, 1, batch_size=B, critic_dist_info=INFO51, prioritized_replay=False, memory_size=4)
        p = torch.softmax(torch.from_numpy(rng.randn(B, 51).astype(np.float32) * 3), 1).numpy()
        r = (-60 * rng.rand(B)) if trial % 2 else -rng.randint(0, 3, B).astype(np.float64)
        done = np.zeros(B, bool) if trial < 4 else (rng.rand(B) < 0.3)
        if trial == 5:
            r = -40 * rng.rand(B)      # terminal rows all non-integer, unclamped (no H6 mix)
        for key, v in (("probs", p), ("r", r), ("done", done), ("m", digest(d.reproject2(p, r, done)))):
            proj[key].append(v)
    for key, v in proj.items():
        out["proj_" + key] = np.stack(v)

    rng = np.random.RandomState(6)
    B = 32
    d = ref.ddpg.DDPG(3, 1, batch_size=B, critic_dist_info=INFO51, prioritized_replay=False, memory_size=4, n_steps=5)
    p = torch.softmax(torch.from_numpy(rng.randn(B, 51).astype(np.float32)), 1).numpy()
    r = -3 * rng.rand(B)
    done = np.zeros(B, bool)
    out["h5_probs"], out["h5_r"], out["h5_done"] = p, r, done
    out["h5_m_live"] = digest(d.reproject2(p, r, done))
    out["h5_m_nstep"] = digest(d.reproj_categorical_dist(p.astype(np.float64), r, done.astype(np.float64)), np.float64)

    B, mem, n_fill, steps, seed, data_seed = 48, 700, 650, 5, 21, 22
    a0, c0 = regen_init(seed, 17, 6, 51)          # before make_learner_pair, which reseeds every generator
    g, l, oa, oc = ref_shim.make_learner_pair(17, 6, INFO51, B, mem, seed=seed)
    for k in NAMES:                 # the test rebuilds the initial weights from the seed
        assert torch.equal(a0[k], l.actor.state_dict()[k]) and torch.equal(c0[k], l.critic.state_dict()[k]), k
    rows = transitions(data_seed, n_fill, 17, 6)
    for s, a, r, s2 in rows:
        l.replayBuffer.add(s, a, r, s2, False)
    out["train_meta"] = np.array([B, mem, n_fill, steps, seed, data_seed])
    out["train_data"] = digest(np.concatenate([np.concatenate([s, a, [r], s2]) for s, a, r, s2 in rows]), np.float64)
    us, tree, params = [], [], []
    for t in range(steps):
        random.seed(300 + t)
        st = random.getstate()
        us.append(digest(np.array([random.random() for _ in range(B)]), np.float64))
        random.setstate(st)
        l.train(g)
        tree.append(digest(np.array([float(x) for x in l.replayBuffer._it_sum._value]), np.float64))
        # [step, network (actor, critic, actor_target, critic_target), tensor (NAMES order)]
        params.append([[digest(mod.state_dict()[k]) for k in NAMES]
                       for mod in (l.actor, l.critic, l.actor_target, l.critic_target)])
    out["train_u"], out["train_tree_sum"], out["train_params"] = np.stack(us), np.stack(tree), np.array(params)

    size = 1 << 16
    buf = ref.prioritized_replay_memory.PrioritizedReplayBuffer(size, alpha=0.6)
    z = np.zeros(1, np.float32)
    for i in range(size - 3):
        buf.add(z, z, 0.0, z, False)
    random.seed(5)
    st = random.getstate()
    out["pristine_u"] = digest(np.array([random.random() for _ in range(2000)]), np.float64)
    random.setstate(st)
    out["pristine_idx"] = np.array(buf._sample_proportional(2000), dtype=np.int32)
    np.savez_compressed(os.path.join(HERE, "oracle_vs_reference.npz"), **out)
    print("oracle_vs_reference.npz:", len(out), "arrays")


def main():
    ref = ref_shim.load()
    torch.set_num_threads(1)
    if len(sys.argv) > 1 and sys.argv[1] == "baseline":      # only the BASELINE-size fixtures (added in round 2)
        gen_baseline_sizes(ref)
        return
    if len(sys.argv) > 1 and sys.argv[1] == "nstep":
        gen_nstep(ref)
        return
    if len(sys.argv) > 1 and sys.argv[1] == "oracle_vs_reference":
        gen_oracle_vs_reference(ref)
        return
    gen_projection(ref)
    gen_tree(ref)
    gen_init(ref)
    # config-2 shapes (small batch so fixtures stay small), PER on, 3 steps, 5 % terminal
    gen_train(ref, "per_c2", 17, 6, INFO51, 32, 600, 600, True, 3, 0.05, seed=11)
    # partially filled buffer (len < size, len-1 exclusion visible), no terminals
    gen_train(ref, "per_part", 17, 6, INFO51, 16, 1000, 333, True, 3, 0.0, seed=12)
    # config 1: Pendulum dims, uniform replay_memory.py
    gen_train(ref, "uniform_c1", 3, 1, INFO_PEND, 64, 500, 400, False, 3, 0.0, seed=13)
    gen_baseline_sizes(ref)
    gen_nstep(ref)
    gen_oracle_vs_reference(ref)


if __name__ == "__main__":
    main()
