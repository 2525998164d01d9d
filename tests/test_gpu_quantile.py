"""Quantile regression DQN (QR-DQN) on the GPU: the learn step, act and the host API against tests/quantile_oracle.py,
and the bit-equality invariants of the other learn paths."""
import ctypes as C

import numpy as np
import pytest
import torch

import quantile_oracle as QO
import replay_oracle as O
from oracle.dqn import adam_scalars, adam_update_
from parity_util import RTOL, check_nstep_against_oracle, close, draw_words, fill_rings, host_ring
from test_gpu_dist import backward64, fill, load

pytestmark = pytest.mark.gpu

N_Q = 50


def qr_group(n, cap, b, h=64, a=4, nq=N_Q, kappa=1.0, seed=0, **extra):
    from dmdqn_b200.group import AgentGroup
    cfg = {"nn_layers": [h, h], "replay_buffer_size": cap, "batch_size": b, "learning_rate": 5e-4, "gamma": 0.99,
           "target_update_frequency": 3, "quantile": True, "num_quantiles": nq, "quantile_kappa": kappa}
    cfg.update(extra)
    return AgentGroup(n, cfg, action_size=a, seed=seed)


def pads_are_zero(grp):
    """Head columns a >= A or i >= N of every block (and the gradient block) are exactly 0."""
    L, H, A, n, npad = grp.layout, grp.hidden, grp.action_size, grp.num_quantiles, grp.atom_stride
    for name in ("theta", "theta_tgt", "adam_m", "adam_v", "grads"):
        t = getattr(grp, name)
        w3 = t[:, L.w3:L.w3 + H * 4 * npad].view(-1, H, 4, npad)
        b3 = t[:, L.b3:L.b3 + 4 * npad].view(-1, 4, npad)
        for blk in (w3[:, :, A:], w3[:, :, :, n:], b3[:, A:], b3[:, :, n:]):
            assert not torch.any(blk != 0), f"{name}: a pad column is not 0"


def oracle_for(grp, n, h, a, nq, kappa=1.0, seed=50, **kw):
    stk = QO.QuantileOracle(n, 89, [h, h], a, nq, kappa, gamma=0.99, learning_rate=5e-4, target_update_frequency=3,
                            seed0=seed, **kw)
    rng = np.random.default_rng(seed + h + nq)
    for k in (1, 3, 5):
        stk.online[k] += torch.as_tensor(rng.standard_normal(stk.online[k].shape).astype(np.float32)) * 0.05
        stk.target[k].copy_(stk.online[k])
    return stk


def one_step_against_the_oracle(h, a, nq, steps=1, b=64, clip=None, kappa=1.0, **extra):
    n, cap = 3, 200
    grp = qr_group(n, cap, b, h=h, a=a, nq=nq, kappa=kappa, global_clipnorm=clip, **extra)
    double_dqn = extra.get("double_dqn", True)
    stk = oracle_for(grp, n, h, a, nq, kappa, double_dqn=double_dqn)
    load(grp, stk)
    fill(grp, [cap + 40, 150, cap], seed=h + nq)
    ring = host_ring(grp)
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    rng = np.random.default_rng(h + a + nq)
    prioritized, n_step = grp.prioritized, grp.n_step
    checked = 0
    for step in range(steps):
        th0 = [torch.stack(x) for x in zip(*[grp.get_weights(i, "online") for i in range(n)])]
        m0 = [torch.stack(x) for x in zip(*[grp.get_weights(i, "m") for i in range(n)])]
        v0 = [torch.stack(x) for x in zip(*[grp.get_weights(i, "v") for i in range(n)])]
        tg0 = grp.theta_tgt.clone()
        for p, q in zip(stk.online, th0):
            p.copy_(q)
        for p, q in zip(stk.target, [torch.stack(x) for x in zip(*[grp.get_weights(i, "target") for i in range(n)])]):
            p.copy_(q)
        if prioritized:
            pr0 = grp.priority.cpu().numpy()
        metrics = grp.learn(draw_words(rng, n, b)).cpu().numpy()
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        gblk = grp.grads.clone()
        slots, nslots = dbg["rows"] % cap, dbg["next_rows"] % cap
        outs = check_nstep_against_oracle(grp, ring, dbg, n_step, what=f"step {step}")
        take = lambda arr, s: np.stack([arr[g, s[g]] for g in range(n)])
        S, A_, S2 = take(obs, slots), take(act, slots), take(nobs, nslots)
        Rn, disc = (np.stack([o[k] for o in outs]) for k in ("r_hat", "discount"))
        isw = dbg["is_weights"] if prioritized else None
        out = stk.learn_on_batch(S, A_, Rn, S2, None, is_weights=isw, discounts=disc, apply=False)
        # expected Q views (0 past A), rows whose a* is a near-tie excluded from the targets and what follows them
        for key in ("q_all", "q_next", "tq_all"):
            close(dbg[key][..., :a], out[key], what=f"step {step} {key}")
            assert not np.any(dbg[key][..., a:] != 0)
        sel = np.sort(out["q_next"] if double_dqn else out["tq_all"], axis=2)
        tie = (sel[..., -1] - sel[..., -2]) < 4 * RTOL * np.abs(sel).max() if a > 1 else np.zeros(sel.shape[:2], bool)
        assert tie.mean() < 0.1
        t = dbg["target_dist"]
        close(t[..., :nq][~tie], out["T"][~tie], what=f"step {step} target samples")
        assert not np.any(t[..., nq:] != 0)
        # the logit gradient, then the parameter gradients in float64 from the kernel's own logit gradient on the kernel's
        # ReLU branch
        npad = grp.atom_stride
        dxd = dbg["dlogits"].reshape(n, b, 4, npad)
        assert not np.any(dxd[:, :, a:] != 0) and not np.any(dxd[..., nq:] != 0)
        dxd = dxd[:, :, :a, :nq].reshape(n, b, a * nq)
        close(dxd[~tie], out["dlogits"].reshape(n, b, -1)[~tie], what=f"step {step} logit gradient")
        g64 = backward64([p.numpy() for p in th0], S, dxd, dbg["dh1"] != 0, dbg["dh2"] != 0)
        # the metrics row: weighted batch-mean loss, Q mean / std over a < A, histogram, learned flag
        qa = out["q_all"].astype(np.float64).reshape(n, -1)
        hist = np.stack([np.bincount(A_[g], minlength=4) for g in range(n)])
        close(metrics[:, 1], qa.mean(1), scale=np.abs(qa).max(), what="q mean")
        close(metrics[:, 2], qa.std(1), scale=np.abs(qa).max(), rtol=1e-4, what="q std")
        assert np.array_equal(metrics[:, 3:7], hist) and np.all(metrics[:, 7] == 1)
        if prioritized:                                 # the unweighted loss of each row, from the device's own terms
            pr1 = grp.priority.cpu().numpy()
            for g in range(n):
                if tie[g].any():
                    continue
                ref = O.priority_of(out["row_loss"][g], 0.6, 1e-6)
                close(pr1[g, slots[g]], ref, what=f"step {step} net {g}: priorities")
                untouched = np.ones(cap, bool); untouched[slots[g]] = False
                assert np.array_equal(pr1[g, untouched], pr0[g, untouched])
            assert np.all(grp.priority_max.cpu().numpy() >= pr1.max(1))
        alpha_t, eps_t = adam_scalars(int(grp.learn_step_host[0]), 5e-4, "keras")
        for i in range(n):
            if not tie[i].any():
                checked += 1
                close(metrics[i, 0], out["loss"][i], what=f"step {step} net {i} loss")
            got = grp.unpack(gblk[i])
            for k in range(6):
                close(got[k].numpy(), g64[k][i], what=f"step {step} net {i} grad[{k}]")
            # Adam on the device's gradient (scaled when clipping): theta, m, v
            g_all = [x.clone() for x in got]
            if clip is not None:
                nrm = float(np.sqrt(sum(float((x.double() ** 2).sum()) for x in g_all)))
                close(grp.grad_norms.cpu().numpy()[i], nrm, what="norm")
                s = np.float32(clip / max(nrm, clip))
                if s != 1:
                    g_all = [x * s for x in g_all]
            th, mm, vv = grp.get_weights(i, "online"), grp.get_weights(i, "m"), grp.get_weights(i, "v")
            for k in range(6):
                p, m_, v_ = th0[k][i].clone(), m0[k][i].clone(), v0[k][i].clone()
                adam_update_(p, g_all[k], m_, v_, alpha_t, eps_t)
                close(th[k].numpy(), p.numpy(), what=f"step {step} net {i} theta[{k}]")
                close(mm[k].numpy(), m_.numpy(), what=f"step {step} net {i} m[{k}]")
                close(vv[k].numpy(), v_.numpy(), rtol=2 * RTOL, what=f"step {step} net {i} v[{k}]")
        # the target sync: hard every 3 steps, or Polyak every step
        ls = int(grp.learn_step_host[0])
        if extra.get("tau") is not None:
            tau = float(np.float32(extra["tau"]))
            close(grp.theta_tgt.cpu().numpy(), (tau * grp.theta + (1.0 - tau) * tg0).cpu().numpy(), what="polyak")
        elif ls % 3 == 0:
            assert torch.equal(grp.theta_tgt, grp.theta)
        else:
            assert torch.equal(grp.theta_tgt, tg0)
        pads_are_zero(grp)
    assert checked > 0
    return grp


@pytest.mark.parametrize("h,a,nq", [(64, 2, 2), (64, 4, 50), (128, 3, 11), (256, 4, 50), (256, 2, 64), (512, 4, 64)])
def test_one_step_matches_the_oracle(h, a, nq):
    one_step_against_the_oracle(h, a, nq)


@pytest.mark.parametrize("extra", [{"sample_mode": "prioritized"}, {"n_step": 3}, {"double_dqn": False}, {"tau": 0.05},
                                   {"clip": 0.05}, {"clip": 1e6}, {"kappa": 0.0}])
def test_learn_variants_match_the_oracle(extra):
    one_step_against_the_oracle(128, 4, N_Q, steps=4, **extra)


def test_free_running_steps_against_the_oracle():
    """30 steps, the oracle's state reset to the device's before each (so every step checks the kernels)."""
    one_step_against_the_oracle(64, 4, 11, steps=30, b=32)


def test_act_matches_the_oracle_and_skips_exploring_agents():
    n, h, a, nq = 64, 128, 3, N_Q
    grp = qr_group(n, 100, 32, h=h, a=a, nq=nq)
    stk = oracle_for(grp, n, h, a, nq)
    load(grp, stk)
    rng = np.random.default_rng(3)
    obs = rng.integers(-1, 20, (n, 89)).astype(np.float32)
    acts, q = grp.act(obs, return_q=True)
    ref_a, ref_q = stk.act(obs, np.zeros(n), np.zeros(n, np.uint32), np.zeros(n, np.uint32))
    q = q.cpu().numpy()
    close(q[:, :a], ref_q, what="expected Q")
    assert not np.any(q[:, a:] != 0)
    srt = np.sort(ref_q, 1)
    ok = (srt[:, -1] - srt[:, -2]) > 4 * RTOL * np.abs(ref_q).max()
    assert ok.mean() > 0.9 and np.array_equal(acts.cpu().numpy()[ok], ref_a[ok])
    eps = np.where(np.arange(n) % 2 == 0, 1.0, 0.0)
    acts2, q2 = grp.act(obs, eps=eps, return_q=True)
    q2 = q2.cpu().numpy()
    assert np.all(np.isnan(q2[::2])) and np.array_equal(q2[1::2], q[1::2])
    assert np.array_equal(acts2.cpu().numpy()[1::2], acts.cpu().numpy()[1::2])
    assert np.all(acts2.cpu().numpy() < a)


def _twins(n=6, cap=200, b=64, **extra):
    a, c = (qr_group(n, cap, b, h=128, seed=7, **extra) for _ in range(2))
    for g in (a, c):
        fill(g, cap, seed=8)
    return a, c


STATE = ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step", "metrics")


@pytest.mark.parametrize("extra", [{}, {"sample_mode": "prioritized"}])
def test_captured_learn_equals_plain_learn(extra):
    a, c = _twins(**extra)
    replay, draws = c.capture_learn()
    a.learn(draws.clone())
    rng = np.random.default_rng(9)
    for it in range(4):
        w = draw_words(rng, 6, 64)
        draws.copy_(w)
        replay()
        a.learn(w)
        torch.cuda.synchronize()
        for name in STATE + (("priority",) if a.prioritized else ()):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name}"


def test_captured_step_host_equals_step_host():
    n, b = 6, 64
    a, c = _twins(n=n, b=b)
    sa, sc = a.make_step_block(), c.make_step_block()
    rng = np.random.default_rng(13)
    replay = None
    for it in range(4):
        vals = {"obs": rng.integers(-1, 20, (n, 89)).astype(np.float32), "next_obs": rng.integers(-1, 20, (n, 89)).astype(np.float32),
                "act": rng.integers(0, 4, n).astype(np.int32), "rew": -rng.random(n) * 100,
                "done": (rng.random(n) < 0.1).astype(np.uint8),
                "draws": rng.integers(0, 2**32, (n, b), dtype=np.uint64).astype(np.uint32).view(np.int32)}
        for blk in (sa, sc):
            for k, v in vals.items():
                blk["host"][k].copy_(torch.as_tensor(v))
        ma = a.step_host(sa)
        if replay is None:
            replay = c.capture_step_host(sc)
            mc = sc["metrics_host"]
        else:
            mc = replay()
        torch.cuda.synchronize()
        assert torch.equal(ma, mc), f"step {it}: metrics"
        for name in STATE + ("obs",):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name}"


def test_a_network_of_a_group_equals_the_same_network_alone_and_runs_repeat():
    from parity_util import copy_state
    big = qr_group(3, 200, 64, h=256, seed=14)
    fill(big, [205, 200, 64], seed=15)
    alone = qr_group(1, 200, 64, h=256, seed=99)
    copy_state(alone, big, slice(1, 2))
    twin = qr_group(3, 200, 64, h=256, seed=1)
    copy_state(twin, big)
    rng = np.random.default_rng(16)
    for it in range(3):
        w = draw_words(rng, 3, 64)
        big.learn(w)
        twin.learn(w)
        alone.learn(w[1:2].contiguous())
        torch.cuda.synchronize()
        for name in STATE:
            assert torch.equal(getattr(big, name)[1:2], getattr(alone, name)), f"step {it}: {name} (network 1 alone)"
            assert torch.equal(getattr(big, name), getattr(twin, name)), f"step {it}: {name} (two runs)"
        for key in ("target_dist", "dlogits"):
            assert torch.equal(big.debug_views()[key], twin.debug_views()[key]), key


def test_shared_parameter_nccl_path_equals_learn_grads_and_adam_apply():
    from dmdqn_b200 import _native as N
    from dmdqn_b200.parallel import SharedParameterStep
    a, c = (qr_group(4, 100, 64, h=128, seed=21, share_parameters=True) for _ in range(2))
    for g in (a, c):
        fill(g, 100, seed=22)
    step = SharedParameterStep.for_group(a, fused=False)
    with pytest.raises(ValueError, match="quantile"):
        SharedParameterStep.for_group(a, fused=True)
    for it in range(3):
        a._gen.manual_seed(100 + it)
        c._gen.manual_seed(100 + it)
        step.step()
        d = c.draw_words((1, c.batch_size))
        N.check(c.lib.dmdqn_learn_grads_quantile(C.byref(c.dims), C.byref(c.hp), C.byref(c.qr), C.byref(c.replay),
                                                 C.byref(c.nets), d.data_ptr(), None, 64, c.grads.data_ptr(),
                                                 c.metrics.data_ptr(), c.workspace.data_ptr(), c.workspace.numel(), None))
        N.check(c.lib.dmdqn_adam_apply_dist(C.byref(c.dims), C.byref(c.hp), C.byref(c.nets), c.num_quantiles, c.grads.data_ptr(),
                                            0.0, None, c.workspace.data_ptr(), c.workspace.numel(), None))
        torch.cuda.synchronize()
        for name in STATE:
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name}"


def test_inactive_networks_stay_untouched_with_zero_metrics():
    grp = qr_group(3, 200, 64, h=64, seed=2)
    fill(grp, [200, 20, 200], seed=3)                  # network 1 holds fewer than batch transitions
    mask = np.array([1, 1, 0], np.uint8)               # network 2 is masked out
    before = {k: getattr(grp, k).clone() for k in ("theta", "theta_tgt", "adam_m", "adam_v")}
    grp.metrics.fill_(7.0)
    metrics = grp.learn(draw_words(np.random.default_rng(1), 3, 64), mask=mask).cpu().numpy()
    assert np.all(metrics[1:] == 0) and metrics[0, 7] == 1
    for k, v in before.items():
        assert torch.equal(getattr(grp, k)[1:], v[1:]), k
        assert not torch.equal(getattr(grp, k)[0], v[0]) or k == "theta_tgt", k
    pads_are_zero(grp)


def test_weights_round_trip(tmp_path):
    from dmdqn_b200.agent import DQNAgent
    grp = qr_group(2, 100, 32, h=64, a=3, nq=11)
    ws = grp.get_weights(1)
    assert [tuple(w.shape) for w in ws] == [(89, 64), (64,), (64, 64), (64,), (64, 33), (33,)]
    new = [w + 0.25 for w in ws]
    grp.set_weights(0, new, sync_target=True)
    for x, y in zip(grp.get_weights(0), new):
        assert torch.equal(x, y)
    assert torch.equal(grp.theta[0], grp.theta_tgt[0])
    pads_are_zero(grp)
    cfg = {"nn_layers": [64, 64], "replay_buffer_size": 100, "batch_size": 32, "quantile": True, "num_quantiles": 11}
    ag = DQNAgent(89, 3, "a0", cfg)
    ag._g.set_weights(0, new)
    path = str(tmp_path / "m.pt")
    ag.save_model(path)
    other = DQNAgent(89, 3, "a1", cfg)
    assert other.load_model(path)
    for x, y in zip(other._g.get_weights(0), new):
        assert torch.equal(x, y)


@pytest.mark.parametrize("nq", [11, 50])
def test_initial_weights_equal_those_of_a_c51_group(nq):
    from dmdqn_b200.group import AgentGroup
    base = {"nn_layers": [64, 64], "replay_buffer_size": 100, "batch_size": 32}
    q = AgentGroup(3, dict(base, quantile=True, num_quantiles=nq), seed=5)
    c = AgentGroup(3, dict(base, distributional=True, num_atoms=nq), seed=5)
    assert q.layout.stride == c.layout.stride
    for name in ("theta", "theta_tgt"):
        assert torch.equal(getattr(q, name), getattr(c, name)), name


def test_quantile_false_is_bit_identical_to_a_group_without_the_key():
    from dmdqn_b200.group import AgentGroup
    base = {"nn_layers": [128, 128], "replay_buffer_size": 200, "batch_size": 64, "target_update_frequency": 3}
    a = AgentGroup(4, dict(base), seed=3)
    c = AgentGroup(4, dict(base, quantile=False, num_quantiles=11, quantile_kappa=0.0), seed=3)
    for g in (a, c):
        fill_rings(g, 200, seed=4)
    rng = np.random.default_rng(5)
    for it in range(3):
        w = draw_words(rng, 4, 64)
        a.learn(w)
        c.learn(w)
        torch.cuda.synchronize()
        for name in STATE:
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name}"
    assert a.layout.stride == c.layout.stride


@pytest.mark.parametrize("extra", [{}, {"sample_mode": "prioritized", "n_step": 3}])
def test_train_loop_runs_quantile_from_the_config(extra):
    from dmdqn_b200.train import PRESETS, train_agents
    cfg = dict(PRESETS["shipped_train_py"])
    cfg.update(max_sim_time=600.0, backend="fake", grid_rows=3, grid_cols=3, fake_traci_seed=11, batch_size=16,
               nn_layers=[64, 64], precision="auto", quantile=True, num_quantiles=50, **extra)
    history, agents, group = train_agents(cfg, episodes=1, mode="batched", seed=3, learn=True)
    t = len(history)
    assert group.quantile and not group.distributional and group.hp.precision == 0
    assert t > 16 and np.all(group.learn_step.cpu().numpy() == t - 15)
    losses = [h["total_loss"] for h in history]
    assert np.all(np.isfinite(losses)) and any(x != 0 for x in losses)
