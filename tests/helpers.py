"""Shared test helpers: golden-fixture access and the compact-array comparison."""
import hashlib
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
STRIDE = 31          # must match tests/golden/make_golden.py
NAMES = ["fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias",
         "fc2_2.weight", "fc2_2.bias", "fc3.weight", "fc3.bias"]


def load(name):
    return np.load(os.path.join(GOLDEN, name))


def digest(t, dtype=np.float32):
    """SHA-256 of an array's values as `dtype`, as 32 uint8: bit-exact equality for arrays too large to store.  Adding
    +0.0 maps -0.0 to +0.0, so two NaN-free arrays get the same digest exactly when np.array_equal holds for them."""
    a = np.ascontiguousarray(torch.as_tensor(t).detach().cpu().numpy(), dtype=dtype) + dtype(0.0)
    return np.frombuffer(hashlib.sha256(a.tobytes()).digest(), dtype=np.uint8)


class ScriptedEnv(object):
    """Deterministic gym-style env for replay_memory.py:21-59 (Replay.initialize): float32-representable states,
    Python-float rewards, scripted episode lengths (some shorter than n_steps)."""
    LENGTHS = [7, 3, 12, 5, 4, 9, 30]

    class _Space(object):
        shape = (2,)
    action_space = _Space()

    def __init__(self):
        self.ep = -1
        self.log = []                       # per episode: dict of lists

    def reset(self):
        self.ep += 1
        self.t = 0
        self.state = np.array([0.25 * (self.ep + 1), -0.5, 1.0 + self.ep], dtype=np.float32).astype(np.float64)
        self.log.append(dict(s=[], a=[], r=[], s2=[], d=[]))
        return self.state

    def step(self, action):
        a = np.asarray(action, dtype=np.float64)
        nxt = (0.875 * self.state + np.array([a[0], a[1], 0.125 * self.t])).astype(np.float32).astype(np.float64)
        reward = float(-np.abs(self.state).sum() + 0.1 * a[0])
        done = self.t == self.LENGTHS[self.ep % len(self.LENGTHS)] - 1
        e = self.log[-1]
        e["s"].append(self.state.copy()); e["a"].append(a.copy()); e["r"].append(reward); e["s2"].append(nxt.copy()); e["d"].append(done)
        self.state = nxt
        self.t += 1
        return nxt, reward, done, {}


def train_data(g):
    """(S, A, R, S2, D) of a train_*.npz fixture: stored, or -- big fixtures -- regenerated from the seed with the
    recipe of tests/golden/make_golden.py:train_data and checked against the stored subsample / checksums."""
    if "S" in g.files:
        return g["S"], g["A"], g["R"], g["S2"], g["D"]
    obs_dim, act_dim, _, _, _, n_fill = [int(x) for x in g["meta"][:6]]
    rng = np.random.RandomState(int(g["seed"]) + 1)
    S = rng.randn(n_fill, obs_dim).astype(np.float32)
    A = rng.uniform(-1, 1, (n_fill, act_dim)).astype(np.float32)
    R = (-3.0 * rng.rand(n_fill)).astype(np.float32).astype(np.float64)
    S2 = rng.randn(n_fill, obs_dim).astype(np.float32)
    D = rng.rand(n_fill) < float(g["term_p"])
    check_compact(g, "S", S, 0.0)
    check_compact(g, "R", R, 0.0)
    return S, A, R, S2, D


def transitions(seed, n, obs_dim, act_dim):
    """n (s, a, r, s2) rows drawn one at a time from RandomState(seed): f32 states and actions, f32-representable
    Python-float rewards (what an environment loop hands to add())."""
    rng = np.random.RandomState(seed)
    rows = []
    for _ in range(n):
        s = rng.randn(obs_dim).astype(np.float32)
        a = rng.uniform(-1, 1, act_dim).astype(np.float32)
        r = float(np.float32(-3 * rng.rand()))
        s2 = rng.randn(obs_dim).astype(np.float32)
        rows.append((s, a, r, s2))
    return rows


def projection_c5_inputs():
    """Inputs of tests/golden/projection_c5_b4096.npz (B=4096, 101 atoms, n_steps=5), regenerated from its seed with
    the recipe of make_golden.py:gen_baseline_sizes and checked against the stored subsamples."""
    g = load("projection_c5_b4096.npz")
    rng = np.random.RandomState(int(g["seed"]))
    B = int(g["B"])
    z = (rng.randn(B, 101) * 2.0).astype(np.float32)
    p = torch.softmax(torch.from_numpy(z), dim=1).numpy()
    r = (40.0 * (rng.rand(B) - 0.5)).astype(np.float32).astype(np.float64)
    done = rng.rand(B) < 0.05
    check_compact(g, "probs", p, 0.0)
    check_compact(g, "r", r, 0.0)
    assert int(done.sum()) == int(g["done_count"])
    return g, p, r, done


def check_params(g, key, arr, atol=1e-5, outlier_atol=2.5e-4, outlier_frac=0.1, stats=None):
    """Post-Adam parameters / targets / moments.  Adam divides by sqrt(v)+eps, so an element whose
    gradient is ~0 by cancellation turns a 1e-10 gradient difference (any fp32 summation-order
    change, e.g. a different BLAS) into a difference of up to ~lr in the parameter.  Gradients are
    held to 1e-5 absolute AND 1e-4 relative-L2 elsewhere; here: all but `outlier_frac` of the elements
    within `atol`, every element within `outlier_atol` (= lr/4)."""
    arr = np.asarray(arr).reshape(-1)
    if key in g.files:
        ref, mine = g[key].reshape(-1), arr
    else:
        ref, mine = g[key + "__sub"], arr[::STRIDE]
        assert arr.size == int(g[key + "__chk"][2])
    err = np.abs(ref.astype(np.float64) - mine.astype(np.float64))
    assert err.max() <= outlier_atol, "%s: max abs err %.3e > %.1e" % (key, err.max(), outlier_atol)
    bad = float((err > atol).mean())
    assert bad <= outlier_frac, "%s: %.4f of elements differ by more than %.1e" % (key, bad, atol)
    if stats is not None:                    # observed slack, reported by the caller
        stats["param_outlier_frac"] = max(stats.get("param_outlier_frac", 0.0), bad)
        stats["param_max_err"] = max(stats.get("param_max_err", 0.0), float(err.max()))
    return err.max()


def check_compact(g, key, arr, atol, what=""):
    """Compare `arr` with a golden entry stored whole or as subsample+checksums."""
    arr = np.asarray(arr)
    if key in g.files:
        ref = g[key]
        assert ref.size == arr.size, (key, ref.shape, arr.shape)
        ref, arr = ref.reshape(-1), arr.reshape(-1)
        err = np.abs(ref.astype(np.float64) - arr.astype(np.float64)).max() if arr.size else 0.0
        assert err <= atol, "%s %s: max abs err %.3e > %.1e" % (what, key, err, atol)
        return err
    sub, chk = g[key + "__sub"], g[key + "__chk"]
    flat = arr.reshape(-1)
    assert flat.size == int(chk[2]), (key, flat.size, chk[2])
    err = np.abs(sub.astype(np.float64) - flat[::STRIDE].astype(np.float64)).max()
    assert err <= atol, "%s %s: subsample max abs err %.3e > %.1e" % (what, key, err, atol)
    s = flat.astype(np.float64).sum()
    assert abs(s - chk[0]) <= atol * flat.size, "%s %s: checksum %.6e vs %.6e" % (what, key, s, chk[0])
    return err


def regen_init(seed, obs_dim, act_dim, n_atoms):
    """Initial actor/critic weights of a train_*.npz fixture, regenerated from its
    seed with the oracle's RNG-parity initialisers (global DDPG is built first:
    actor, actor_target, critic, ... -- ddpg.py:56-64)."""
    import random
    from oracle import d4pg_oracle as O
    torch.manual_seed(seed)
    np.random.seed(seed)
    random.seed(seed)
    a = O.init_actor(obs_dim, act_dim)
    O.init_actor(obs_dim, act_dim)               # actor_target consumes the RNG too
    c = O.init_critic(obs_dim, act_dim, n_atoms)
    return a, c


def assert_tree_close_and_sync(buf, want_sum, want_min, max_mismatch_frac=0.01):
    """Device tree vs reference/oracle tree.  Leaves are `np.float32 ** 0.6` in the reference, i.e.
    the host libm's powf (glibc: <=0.82 ULP, not correctly rounded, and its FMA/non-FMA ifunc
    variants differ), so leaf parity is: every leaf within 1 ulp, all but 1% bit-equal.  Internal
    nodes are then compared after substituting the reference leaves, and the device trees are
    overwritten with the reference trees so that *index* parity in later rounds is asserted
    given identical tree contents (SURVEY.md section 7)."""
    import torch
    st = buf._store
    cap = st.capacity
    got = st.sum_tree.cpu().numpy()
    want = np.asarray(want_sum, dtype=np.float32)
    gl, wl = got[cap:], want[cap:]
    ulp = np.spacing(np.abs(wl).astype(np.float32))
    assert (np.abs(gl.astype(np.float64) - wl.astype(np.float64)) <= ulp).all(), "leaf off by more than 1 ulp"
    touched = max(1, int((wl != 1.0).sum()))
    mism = int((gl != wl).sum())
    assert mism <= max(1, max_mismatch_frac * touched), "%d of %d leaves differ" % (mism, touched)
    if mism == 0:
        assert np.array_equal(got, want), "internal nodes differ although all leaves match"
        assert np.array_equal(st.min_tree.cpu().numpy(), np.asarray(want_min, dtype=np.float32))
    st.sum_tree.copy_(torch.from_numpy(want))
    st.min_tree.copy_(torch.from_numpy(np.asarray(want_min, dtype=np.float32)))
    return mism


def rel_l2(mine, ref):
    mine, ref = np.asarray(mine, np.float64).reshape(-1), np.asarray(ref, np.float64).reshape(-1)
    return float(np.linalg.norm(mine - ref) / max(np.linalg.norm(ref), 1e-30))


def golden_vec(g, key, arr):
    """(reference values, matching slice of arr) for whole or subsampled fixtures."""
    arr = np.asarray(arr).reshape(-1)
    if key in g.files:
        return g[key].reshape(-1), arr
    return g[key + "__sub"], arr[::STRIDE]
