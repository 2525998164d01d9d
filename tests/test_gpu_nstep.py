"""n-step returns on the GPU (n_step > 1) against tests/replay_oracle.py: the sampled returns, discounts and bootstrap rows
(bit-exact, every sample mode, n_step 1 included), the unchanged one-step path, learn parity, prioritized replay and
shared parameters with n-step targets, and the execution orders that must not change a bit, with and without prioritized
replay.  The bodies shared with the prioritized-replay tests live in tests/parity_util.py.  Run on the B200 box:
pytest -m gpu"""
import numpy as np
import pytest
import torch

import replay_oracle as O
from oracle import replay as R
from parity_util import (NSTEP, PER, captured_learn_equals_plain_learn, captured_step_host_equals_step_host,
                         chained_step_equals_stage_by_stage_step, check_nstep_against_oracle, close, draw_words, fill_rings,
                         host_ring, learn_matches_the_oracle, one_group_of_eight_equals_two_groups_of_four, replay_group,
                         train_loop_learns_from_the_config_alone)

pytestmark = pytest.mark.gpu
NSTEP_CONFIGS = (NSTEP, {**PER, **NSTEP})             # the execution orders hold with and without prioritized replay


# ------------------------------------------------------------------ 1. sampling -----------------------------------------
N_WRITTEN = np.array([256, 300, 1000, 5000, 12345, 20000, 29999, 30000, 30001, 45678, 60000, 384, 777, 4096, 29000, 100000])


@pytest.mark.parametrize("n", [1, 3, 8])
@pytest.mark.parametrize("mode", ["fisher_yates", "replacement", "indices", "prioritized"])
def test_sampling_is_bit_exact_against_the_oracle(mode, n):
    """Returns, discounts, terminal flags and bootstrap rows; at n = 1 these are the one-step targets on the drawn rows."""
    cap, b = 30000, 256
    grp = replay_group(16, cap, b, n_step=n, sample_mode=mode)
    fill_rings(grp, N_WRITTEN, seed=1)
    ring = host_ring(grp)
    size = np.minimum(N_WRITTEN, cap)
    nobs = grp.next_obs.cpu().numpy()[..., :89]
    pr = grp.priority.cpu().numpy() if grp.priority is not None else None
    rng = np.random.default_rng(2)
    for it in range(2):
        if mode == "indices":                          # the newest rows of every ring, then random ones
            draws = np.stack([np.concatenate([size[g] - 1 - np.arange(16), rng.integers(0, size[g], b - 16)])
                              for g in range(16)]).astype(np.int32)
            dev = torch.as_tensor(draws).cuda()
        else:
            dev = draw_words(rng, 16, b)
            draws = dev.cpu().numpy().view(np.uint32)
        states, actions, rewards, next_states, dones, active = grp.sample(dev)
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        for g in range(16):
            if mode == "prioritized":
                slots = O.prioritized_indices(pr[g], draws[g])
            else:
                logical = {"fisher_yates": lambda: R.fisher_yates_indices(draws[g], size[g]),
                           "replacement": lambda: R.replacement_indices(draws[g], size[g]),
                           "indices": lambda: draws[g]}[mode]()
                slots = ring.logical_to_slot(g, logical)
            assert np.array_equal(dbg["rows"][g], g * cap + slots), f"{mode} call {it} agent {g}: rows"
        outs = check_nstep_against_oracle(grp, ring, dbg, n, what=f"{mode} call {it}")
        if n == 1:
            assert all(np.all(o["m"] == 1) for o in outs) and np.array_equal(dbg["next_rows"], dbg["rows"])
        else:
            assert any(o["m"].min() < n for o in outs) and all(o["m"].max() <= n for o in outs)
        dones_ref = np.stack([o["done"] for o in outs])
        assert np.array_equal(dones.cpu().numpy(), dones_ref) and np.array_equal(rewards.cpu().numpy(), dbg["r_hat"])
        nref = np.stack([nobs[g, dbg["next_rows"][g] - g * cap] for g in range(16)])
        assert np.array_equal(next_states.cpu().numpy(), nref), f"{mode} call {it}: gathered next states"
        assert np.all(active.cpu().numpy() == 1)
        if mode == "indices":                          # the newest row of every ring bootstraps from itself
            assert np.all(dbg["next_rows"][:, 0] == dbg["rows"][:, 0])


# ------------------------------------------------------------------ 2. one-step path ------------------------------------
@pytest.mark.parametrize("precision,h", [("fp32", 64), ("tf32x3", 256)])
@pytest.mark.parametrize("mode", ["fisher_yates", "prioritized"])
def test_n_step_one_and_zero_are_the_one_step_path_bit_for_bit(precision, h, mode):
    from dmdqn_b200.group import AgentGroup
    n, cap, b = 6, 300, 64
    base = {"nn_layers": [h, h], "replay_buffer_size": cap, "batch_size": b, "learning_rate": 5e-4, "gamma": 0.99,
            "target_update_frequency": 3, "precision": precision, "sample_mode": mode}
    plain = AgentGroup(n, base, seed=4)
    one = AgentGroup(n, dict(base, n_step=1), seed=4)
    zero = AgentGroup(n, dict(base, n_step=1), seed=4)
    zero.hp.n_step = 0                                 # what a zero-initialised C caller passes
    groups = (plain, one, zero)
    for grp in groups:
        fill_rings(grp, [cap + 17, cap, 200, 64, 1000, 150], seed=6, done_rate=0.2)
    rng = np.random.default_rng(7)
    for step in range(4):
        w = draw_words(rng, n, b)
        ms = [grp.learn(w).clone() for grp in groups]
        torch.cuda.synchronize()
        dbg = [grp.debug_views() for grp in groups]
        for k in (1, 2):
            assert torch.equal(ms[0], ms[k]), f"step {step} group {k}: metrics"
            assert torch.equal(dbg[0]["y"], dbg[k]["y"]) and torch.equal(dbg[0]["rows"], dbg[k]["next_rows"])
            for name in ("theta", "theta_tgt", "adam_m", "adam_v", "priority", "priority_max"):
                a, c = getattr(plain, name), getattr(groups[k], name)
                assert (a is None and c is None) or torch.equal(a, c), f"step {step} group {k}: {name}"


# ------------------------------------------------------------------ 3. learn parity -------------------------------------
@pytest.mark.parametrize("h,precision,loss,double_dqn,mode", [
    (64, "fp32", "mse", True, "fisher_yates"), (64, "fp32", "huber", False, "fisher_yates"),
    (256, "fp32", "mse", False, "fisher_yates"), (256, "fp32", "huber", True, "fisher_yates"),
    (256, "tf32x3", "mse", True, "fisher_yates"), (256, "tf32x3", "huber", False, "fisher_yates"),
    (64, "fp32", "mse", True, "prioritized"), (256, "tf32x3", "huber", True, "prioritized")])
def test_learn_matches_the_n_step_oracle(h, precision, loss, double_dqn, mode):
    learn_matches_the_oracle(h, precision, loss, double_dqn, mode, 3)


# ------------------------------------------------------------------ 4. shared parameters --------------------------------
def test_shared_parameters_keep_every_lookahead_in_its_own_ring():
    n, cap, b = 6, 120, 256
    grp = replay_group(n, cap, b, share_parameters=True, n_step=5)
    fill_rings(grp, cap + 33, seed=20, done_rate=0.05)
    ring = host_ring(grp)
    stk = O.ReplayStackedOracle(1, 89, [64, 64], 4, gamma=0.99, learning_rate=5e-4, loss="mse", target_update_frequency=3,
                                seed0=7)
    grp.set_weights(0, [p[0] for p in stk.online], "online"); grp.set_weights(0, [p[0] for p in stk.target], "target")
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    rng = np.random.default_rng(21)
    w = draw_words(rng, 1, b)
    grp.learn(w)
    dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
    rows, nrows = dbg["rows"][0], dbg["next_rows"][0]
    logical = R.fisher_yates_indices(w.cpu().numpy().view(np.uint32)[0], cap * n)
    agents = logical // cap
    assert np.array_equal(rows // cap, agents) and np.array_equal(nrows // cap, agents), "a lookahead crossed rings"
    assert np.array_equal(rows % cap, [ring.logical_to_slot(a, np.array([j]))[0] for a, j in zip(agents, logical % cap)])
    (o,) = check_nstep_against_oracle(grp, ring, dbg, 5, what="shared")
    assert o["m"].min() < 5 and o["m"].max() == 5
    out = stk.learn_on_batch(obs[agents, rows % cap][None], act[agents, rows % cap][None], o["r_hat"][None],
                             nobs[agents, nrows % cap][None], o["done"][None], discounts=o["discount"][None])
    close(dbg["y"], out["y"], what="shared TD target")
    close(dbg["q_all"], out["q_all"], what="shared online Q(s)")


# ------------------------------------------------------------------ 5. execution order ----------------------------------
def test_chained_step_equals_stage_by_stage_step():
    for config in NSTEP_CONFIGS:
        chained_step_equals_stage_by_stage_step(config)


def test_captured_learn_equals_plain_learn():
    for config in NSTEP_CONFIGS:
        captured_learn_equals_plain_learn(config)


def test_captured_step_host_equals_step_host():
    for config in NSTEP_CONFIGS:
        captured_step_host_equals_step_host(config)


def test_one_group_of_eight_equals_two_groups_of_four():
    for config in NSTEP_CONFIGS:
        one_group_of_eight_equals_two_groups_of_four(config)


# ------------------------------------------------------------------ the training loop -----------------------------------
@pytest.mark.parametrize("mode", ["batched", "per_agent"])
def test_train_loop_learns_with_n_step_returns_from_the_config_alone(mode):
    train_loop_learns_from_the_config_alone(NSTEP, mode)
