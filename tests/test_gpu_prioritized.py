"""Prioritized replay on the GPU (sample_mode "prioritized") against tests/replay_oracle.py: the push rule, the drawn slots
(bit-exact), the importance weights, the weighted learn step and its priority update, equivalence with the uniform path
when every weight is 1, and the execution orders that must not change a bit.  The bodies shared with the n-step tests
live in tests/parity_util.py.  Run on the B200 box: pytest -m gpu"""
import numpy as np
import pytest
import torch

import replay_oracle as O
from parity_util import (PER, captured_learn_equals_plain_learn, captured_step_host_equals_step_host,
                         chained_step_equals_stage_by_stage_step, draw_words, fill_rings, learn_matches_the_oracle,
                         one_group_of_eight_equals_two_groups_of_four, replay_group, train_loop_learns_from_the_config_alone,
                         ulps)
from oracle import replay as R

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------ 1. push ---------------------------------------------
def test_push_gives_new_slots_the_maximum_priority():
    n, cap = 4, 5
    grp = replay_group(n, cap, 2, **PER)
    ring = O.PrioritizedRing(n, cap, 89)
    rng = np.random.default_rng(0)
    for t in range(13):
        if t in (3, 8):                                # the ring's maximum moves (as the learn step would move it)
            pm = rng.uniform(0.5, 4.0, n).astype(np.float32)
            grp.priority_max.copy_(torch.as_tensor(pm)); ring.priority_max[:] = pm
        mask = (rng.random(n) < 0.7).astype(np.uint8)
        s = rng.integers(-1, 20, (n, 89)).astype(np.float32)
        a, r, dn = rng.integers(0, 4, n).astype(np.int32), rng.random(n), np.zeros(n, bool)
        grp.push(s, a, r, s, dn, mask=mask); ring.push(s, a, r, s, dn, mask=mask)
        assert np.array_equal(grp.priority.cpu().numpy(), ring.priority), f"push {t}"
    assert np.array_equal(grp.n_written.cpu().numpy(), ring.n_written) and ring.n_written.max() > cap   # wrapped around
    assert np.array_equal(grp.priority_max.cpu().numpy(), ring.priority_max)


# ------------------------------------------------------------------ 2. sampling -----------------------------------------
N_WRITTEN = np.array([256, 300, 1000, 5000, 12345, 20000, 29999, 30000, 30001, 45678, 60000, 384, 777, 4096, 29000, 100000])


def test_sampling_is_bit_exact_against_the_oracle():
    n, cap, b = 16, 30000, 256
    grp = replay_group(n, cap, b, per_beta=0.45, **PER)
    fill_rings(grp, N_WRITTEN, seed=1)
    rng = np.random.default_rng(2)
    pr = grp.priority.cpu().numpy()
    rew = grp.rew_ring.cpu().numpy()
    for it in range(3):
        words = draw_words(rng, n, b)
        grp.sample(words)
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        w = words.cpu().numpy().view(np.uint32)
        for g in range(n):
            slots = O.prioritized_indices(pr[g], w[g])
            assert np.array_equal(dbg["rows"][g], g * cap + slots), f"call {it} agent {g}: drawn slots differ"
            assert np.all(slots < min(N_WRITTEN[g], cap))
            ref = O.is_weights(pr[g], slots, 0.45)     # sample() does not advance learn_step: beta_t = beta0
            assert ulps(dbg["is_weights"][g], ref).max() <= 2, f"call {it} agent {g}: importance weights"
            assert np.array_equal(dbg["r_hat"][g], R.zscore_canonical(rew[g, slots]).astype(np.float32))


# ------------------------------------------------------------------ 3. frequencies --------------------------------------
def test_device_frequencies_are_proportional_to_priority():
    from scipy import stats
    n, cap, b, calls = 2, 300, 64, 300
    grp = replay_group(n, cap, b, **PER)
    fill_rings(grp, cap, seed=3)
    grp.priority[:, :40] = 0
    grp.priority[1, 100:110] *= 20
    pr = grp.priority.cpu().numpy().astype(np.float64)
    rng = np.random.default_rng(4)
    hist = np.zeros((n, cap))
    for _ in range(calls):
        grp.sample(draw_words(rng, n, b))
        rows = grp.debug_views()["rows"].cpu().numpy()
        for g in range(n):
            hist[g] += np.bincount(rows[g] - g * cap, minlength=cap)
    for g in range(n):
        assert hist[g, :40].sum() == 0
        expected = pr[g, 40:] / pr[g].sum() * hist[g].sum()
        assert stats.chisquare(hist[g, 40:], expected).pvalue > 1e-4


# ------------------------------------------------------------------ 4. learn parity -------------------------------------
@pytest.mark.parametrize("h,precision,loss", [(64, "fp32", "mse"), (64, "fp32", "huber"), (256, "fp32", "mse"),
                                              (256, "tf32x3", "mse"), (256, "tf32x3", "huber")])
def test_learn_matches_the_weighted_oracle(h, precision, loss):
    learn_matches_the_oracle(h, precision, loss, True, "prioritized", 1)


# ------------------------------------------------------------------ 5. equivalence with uniform -------------------------
@pytest.mark.parametrize("h,precision", [(64, "fp32"), (256, "tf32x3")])
def test_alpha_zero_equals_the_uniform_path_on_the_same_rows(h, precision):
    n, cap, b = 5, 300, 64
    per = replay_group(n, cap, b, h=h, precision=precision, seed=4, per_alpha=0.0, **PER)
    uni = replay_group(n, cap, b, h=h, precision=precision, seed=4, sample_mode="indices")
    for g in (per, uni):
        fill_rings(g, [cap + 17, cap, 200, 64, 1000], seed=6, priorities=False)
    per.priority.copy_((torch.arange(cap, device="cuda")[None, :] < torch.as_tensor(per.sizes_host(), device="cuda")[:, None]).float())
    rng = np.random.default_rng(7)
    nw = per.n_written_host.copy()
    for step in range(4):
        mp = per.learn(draw_words(rng, n, b)).clone()
        dbg = per.debug_views()
        assert torch.all(dbg["is_weights"] == 1.0)
        slots = dbg["rows"].cpu().numpy() - np.arange(n)[:, None] * cap
        size = np.minimum(nw, cap)
        logical = (slots - (nw - size)[:, None]) % cap
        mu = uni.learn(logical.astype(np.int32)).clone()
        torch.cuda.synchronize()
        assert torch.equal(mp, mu), f"step {step}: metrics differ"
        for name in ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step"):
            assert torch.equal(getattr(per, name), getattr(uni, name)), f"step {step}: {name} differs"
        written = torch.as_tensor(per.sizes_host(), device="cuda")[:, None] > torch.arange(cap, device="cuda")[None, :]
        assert torch.all(per.priority[written] == 1.0) and torch.all(per.priority[~written] == 0.0)


# ------------------------------------------------------------------ 6. execution order ----------------------------------
def test_chained_step_equals_stage_by_stage_step():
    chained_step_equals_stage_by_stage_step(PER)


def test_captured_learn_equals_plain_learn_while_beta_anneals():
    captured_learn_equals_plain_learn(PER)


def test_captured_step_host_equals_step_host():
    captured_step_host_equals_step_host(PER)


def test_one_group_of_eight_equals_two_groups_of_four():
    one_group_of_eight_equals_two_groups_of_four(PER)


# ------------------------------------------------------------------ 8. duplicates ---------------------------------------
@pytest.mark.parametrize("h,precision", [(64, "fp32"), (256, "tf32x3")])
def test_a_slot_drawn_twice_keeps_the_priority_of_either_row(h, precision):
    n, cap, b, alpha, eps = 2, 200, 64, 0.7, 1e-6
    grp = replay_group(n, cap, b, h=h, precision=precision, per_alpha=alpha, per_eps=eps, **PER)
    fill_rings(grp, cap, seed=17)
    grp.priority[:, 10] = 1e4                          # slot 10 carries most of the mass: drawn many times per batch
    grp.priority[:, 11] = 5e3
    grp.learn(draw_words(np.random.default_rng(18), n, b))
    dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
    pr = grp.priority.cpu().numpy()
    act = np.stack([grp.act_ring.cpu().numpy()[g, dbg["rows"][g] - g * cap] for g in range(n)])
    delta = np.take_along_axis(dbg["q_all"], act[..., None].astype(np.int64), 2)[..., 0] - dbg["y"]
    for g in range(n):
        slots = dbg["rows"][g] - g * cap
        for s in (10, 11):
            rows = np.nonzero(slots == s)[0]
            assert rows.size >= 2
            assert np.all(delta[g, rows] == delta[g, rows[0]])      # one transition, one TD error
            assert ulps(pr[g, s], O.priority_of(delta[g, rows[:1]], alpha, eps)).max() <= 1


# ------------------------------------------------------------------ the training loop -----------------------------------
@pytest.mark.parametrize("mode", ["batched", "per_agent"])
def test_train_loop_runs_prioritized_from_the_config_alone(mode):
    train_loop_learns_from_the_config_alone(PER, mode)
