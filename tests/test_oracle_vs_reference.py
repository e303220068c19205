"""oracle/ vs the unmodified reference beyond the training fixtures: random projections, the H5 discount, five
DDPG.train() steps and pristine-tree sampling, against the reference's outputs in tests/golden/oracle_vs_reference.npz
(tests/golden/make_golden.py:gen_oracle_vs_reference).  CPU only; runs everywhere."""
import random

import numpy as np
import torch

from oracle import d4pg_oracle as O
from tests import helpers as H

INFO = {"type": "categorical", "v_min": -50.0, "v_max": 0.0, "n_atoms": 51}
FIXTURE = "oracle_vs_reference.npz"


def _uniforms(seed, n):
    random.seed(seed)
    return [random.random() for _ in range(n)]


def test_projection_random_vs_reproject2():
    g = H.load(FIXTURE)
    for trial in range(len(g["proj_m"])):
        m = O.project_live(g["proj_probs"][trial], g["proj_r"][trial], g["proj_done"][trial], -50.0, 0.0, 51, 0.99)
        assert np.array_equal(H.digest(m), g["proj_m"][trial]), trial


def test_h5_live_projection_ignores_n_steps():
    """SURVEY H5: reproject2 discounts with gamma, reproj_categorical_dist with gamma**n."""
    g = H.load(FIXTURE)
    p, r, done = g["h5_probs"], g["h5_r"], g["h5_done"]
    m1 = O.project_live(p, r, done, -50.0, 0.0, 51, 0.99)
    assert np.array_equal(H.digest(m1), g["h5_m_live"])
    m5 = O.project_nstep(p, r, done, -50.0, 0.0, 51, 0.99, 5)
    assert np.array_equal(H.digest(m5, np.float64), g["h5_m_nstep"])
    assert np.abs(m5 - m1).max() > 0.05


def test_five_train_steps_vs_live_reference():
    g = H.load(FIXTURE)
    B, mem, n_fill, steps, seed, data_seed = [int(x) for x in g["train_meta"]]
    a0, c0 = H.regen_init(seed, 17, 6, 51)
    rows = H.transitions(data_seed, n_fill, 17, 6)
    assert np.array_equal(H.digest(np.concatenate([np.concatenate([s, a, [r], s2]) for s, a, r, s2 in rows]), np.float64),
                          g["train_data"]), "regenerated transitions differ from the reference run's"
    buf = O.PrioritizedReplayOracle(mem, 0.6, 17, 6)
    for s, a, r, s2 in rows:
        buf.add(s, a, r, s2, False)
    lo = O.LearnerOracle(17, 6, INFO, actor_w=a0, critic_w=c0)
    sched = O.LinearScheduleOracle(100000, 1.0, 0.4)
    torch.set_num_threads(1)
    for t in range(steps):
        us = _uniforms(300 + t, B)
        assert np.array_equal(H.digest(np.array(us), np.float64), g["train_u"][t])
        batch = buf.sample(B, sched.value(), us)
        out = lo.train_step(*batch[:5])
        buf.update_priorities(batch[6], out["prio"])
        assert np.array_equal(H.digest(buf.sum.value, np.float64), g["train_tree_sum"][t]), t
        for n, (net, mine) in enumerate((("actor", lo.actor), ("critic", lo.critic),
                                         ("actor_target", lo.actor_target), ("critic_target", lo.critic_target))):
            for j, k in enumerate(H.NAMES):
                assert np.array_equal(H.digest(mine[k]), g["train_params"][t, n, j]), (t, net, k)


def test_pristine_tree_sampling_is_f64_at_scale():
    """Before any update_priorities the reference tree holds Python floats: mass = u*sum and the
    descent run in f64.  Needs a buffer large enough that f32 rounding of the mass would matter."""
    g = H.load(FIXTURE)
    size = 1 << 16
    ob = O.PrioritizedReplayOracle(size, 0.6, 1, 1)
    ob.add_batch(np.zeros((size - 3, 1), np.float32), np.zeros((size - 3, 1), np.float32), np.zeros(size - 3),
                 np.zeros((size - 3, 1), np.float32), np.zeros(size - 3, bool))
    us = _uniforms(5, 2000)
    assert np.array_equal(H.digest(np.array(us), np.float64), g["pristine_u"])
    idx_ref = [int(i) for i in g["pristine_idx"]]
    idx = ob.sample_indices(us)
    assert list(idx) == idx_ref
    f32_idx = [O.find_prefixsum_idx(ob.sum.value, ob.capacity, np.float32(np.float32(u) * ob.sum.reduce_prefix(ob.length - 2)))
               for u in us]
    assert f32_idx != idx_ref          # the f32 rule really is different at this size
