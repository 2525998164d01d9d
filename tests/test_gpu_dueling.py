"""Dueling Q-networks on the GPU (config ``dueling``): the fold kernel bit for bit against numpy; the plumbing bit for bit
against a plain group whose head is the folded one (both learn paths, act, the gradient block); the semantics against the
textbook two-stream oracle (tests/dueling_oracle.py); prioritized replay, n-step targets and clipping with dueling heads;
the execution-order invariants; and ``dueling: false`` against a group without the key.  Run on the B200 box: pytest -m gpu"""
import ctypes as C

import numpy as np
import pytest
import torch

from dueling_oracle import DuelingStackedOracle, fold_np, project_np
from oracle.dqn import adam_scalars
from parity_util import (NSTEP, PER, RTOL, adam_close, captured_learn_equals_plain_learn, captured_step_host_equals_step_host,
                         chained_step_equals_stage_by_stage_step, close, draw_words, fill_rings,
                         one_group_of_eight_equals_two_groups_of_four, ulps)

pytestmark = pytest.mark.gpu
DUEL = {"dueling": True}
RING = ("obs", "next_obs", "act_ring", "rew_ring", "done_ring", "n_written", "priority", "priority_max")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _group(n, cap, b, h=64, precision="fp32", a=4, seed=0, **extra):
    from dmdqn_b200.group import AgentGroup
    cfg = {"nn_layers": [h, h], "replay_buffer_size": cap, "batch_size": b, "learning_rate": 5e-4, "gamma": 0.99,
           "target_update_frequency": 3, "precision": precision}
    cfg.update(extra)
    return AgentGroup(n, cfg, action_size=a, seed=seed)


def _fill(grp, n_written, seed):
    fill_rings(grp, n_written, seed=seed, done_rate=0.1)
    grp.act_ring.remainder_(grp.action_size)


def _perturb(grp, seed):
    """Non-zero biases and value head, and a target that differs from the online network."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    L, H = grp.layout, grp.hidden
    for t, s in ((grp.theta, 0.05), (grp.theta_tgt, 0.07)):
        for lo, hi in ((L.b1, L.b1 + H), (L.b2, L.b2 + H), (L.b3, L.b3 + grp.action_size), (L.wv, L.bv + 1)):
            t[:, lo:hi] += torch.randn((t.shape[0], hi - lo), device="cuda", generator=gen) * s


def _fold_block(grp, blk):
    """W3e [H, 4], b3e [4] of one dueling parameter block (numpy fp32 restatement)."""
    L, H = grp.layout, grp.hidden
    b = blk.cpu().numpy()
    return fold_np(b[L.w3:L.w3 + 4 * H].reshape(H, 4), b[L.b3:L.b3 + 4], b[L.wv:L.wv + H], b[L.bv], grp.action_size)


@pytest.mark.parametrize("a", [2, 3, 4])
def test_fold_kernel_writes_the_folded_heads_bit_for_bit(a):
    grp = _group(3, 160, 64, h=128, a=a, **DUEL)
    _perturb(grp, a)
    _fill(grp, 160, seed=a)
    th0, tg0 = grp.theta.clone(), grp.theta_tgt.clone()
    grp.learn(draw_words(np.random.default_rng(a), 3, 64))
    head = grp.debug_views()["head"].cpu().numpy()
    H = grp.hidden
    for which, src in ((0, th0), (1, tg0)):
        for g in range(3):
            w3e, b3e = _fold_block(grp, src[g])
            assert np.array_equal(head[which, g, :4 * H].reshape(H, 4), w3e), (which, g)
            assert np.array_equal(head[which, g, 4 * H:], b3e), (which, g)


def _plain_twin(d):
    """A plain group on the dueling group's rings whose trunk, moments and step counters are the dueling group's and
    whose W3 / b3 (online and target) are the folded heads."""
    p = _group(d.n_agents, d.capacity, d.batch_size, h=d.hidden, precision=d.config["precision"], a=d.action_size,
               sample_mode=d.config["sample_mode"], n_step=d.n_step)
    for name in RING:
        if getattr(d, name) is not None:
            getattr(p, name).copy_(getattr(d, name))
    p.n_written_host[:] = d.n_written_host
    L, H, end = d.layout, d.hidden, int(d.layout.b3) + 4
    for name in ("theta", "theta_tgt", "adam_m", "adam_v"):
        getattr(p, name)[:, :end] = getattr(d, name)[:, :end]
    for name in ("theta", "theta_tgt"):
        for g in range(d.n_nets):
            w3e, b3e = _fold_block(d, getattr(d, name)[g])
            getattr(p, name)[g, L.w3:L.w3 + 4 * H] = torch.as_tensor(w3e.reshape(-1)).cuda()
            getattr(p, name)[g, L.b3:L.b3 + 4] = torch.as_tensor(b3e).cuda()
    p.adam_m[:, L.w3:end] = 0
    p.adam_v[:, L.w3:end] = 0
    d.adam_m[:, L.w3:] = 0
    d.adam_v[:, L.w3:] = 0
    p.learn_step.copy_(d.learn_step); p.learn_step_host[:] = d.learn_step_host
    return p


def _learn_grads(grp, words, grads):
    from dmdqn_b200 import _native as N
    N.check(grp.lib.dmdqn_learn_grads(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.replay), C.byref(grp.nets),
                                      words.data_ptr(), None, grp.batch_size, grads.data_ptr(), grp.metrics.data_ptr(),
                                      grp.workspace.data_ptr(), grp.workspace.numel(), _stream()))


@pytest.mark.parametrize("h,precision,a", [(64, "fp32", 3), (256, "fp32", 4), (256, "tf32x3", 4), (256, "tf32x3", 2)])
def test_dueling_step_equals_a_plain_step_on_the_folded_head(h, precision, a):
    n, cap, b = 4, 200, 128
    d = _group(n, cap, b, h=h, precision=precision, a=a, **DUEL, **PER, **NSTEP)
    _perturb(d, h + a)
    _fill(d, [cap + 30, 170, cap, 140], seed=h)
    saved = {k: getattr(d, k).clone() for k in ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step", "priority",
                                                   "priority_max")}
    p = _plain_twin(d)
    end, L, H = int(d.layout.b3) + 4, d.layout, h
    words = draw_words(np.random.default_rng(h), n, b)
    md, mp = d.learn(words).clone(), p.learn(words).clone()
    dd, dp = d.debug_views(), p.debug_views()
    assert int(dd["tc_error"][0]) == 0 and int(dp["tc_error"][0]) == 0
    assert torch.equal(md, mp)
    for k in ("y", "q_all", "q_next", "tq_all"):
        assert torch.equal(dd[k], dp[k]), k
    assert torch.equal(d.priority, p.priority) and torch.equal(d.priority_max, p.priority_max)
    for name in ("theta", "adam_m", "adam_v", "theta_tgt"):
        assert torch.equal(getattr(d, name)[:, :L.w3], getattr(p, name)[:, :L.w3]), name
    # the gradient block: trunk bit for bit, head = the projection of the plain step's W3 / b3 gradient
    for name, t in saved.items():
        getattr(d, name).copy_(t)
    p2 = _plain_twin(d)
    gd, gp = torch.zeros_like(d.theta), torch.zeros_like(p2.theta)
    _learn_grads(d, words, gd)
    _learn_grads(p2, words, gp)
    torch.cuda.synchronize()
    assert torch.equal(gd[:, :L.w3], gp[:, :L.w3])
    gd, gp = gd.cpu().numpy(), gp.cpu().numpy()
    for g in range(n):
        dw3, db3, dwv, dbv = project_np(gp[g, L.w3:L.w3 + 4 * H].reshape(H, 4), gp[g, L.b3:L.b3 + 4], a)
        assert np.array_equal(gd[g, L.w3:L.w3 + 4 * H].reshape(H, 4), dw3), g
        assert np.array_equal(gd[g, L.b3:L.b3 + 4], db3), g
        assert np.array_equal(gd[g, L.wv:L.wv + H], dwv), g
        assert gd[g, L.bv] == dbv and np.all(gd[g, L.bv + 1:] == 0), g
    # act on the dueling block equals act on the folded plain block
    obs = torch.randn((n, 96), device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    obs[:, 89:] = 0
    ad, qd = d.act(obs, return_q=True)
    ap, qp = p2.act(obs, return_q=True)
    assert torch.equal(ad, ap) and torch.equal(qd, qp)


def _load(grp, stk):
    for i in range(grp.n_nets):
        for which, src in (("online", stk.online), ("target", stk.target), ("m", stk.adam_m), ("v", stk.adam_v)):
            grp.set_weights(i, [p[i] for p in src], which)


def _grads64(params, states, actions, y, mask1, mask2):
    """float64 autograd gradients of the MSE batch-mean loss of the two-stream model at the fp32 parameters ``params``
    against the device's TD targets ``y``, on the piecewise-linear branch the kernel took: relu(z) is z * mask with the
    kernel's relu' masks ``mask1`` / ``mask2`` [N, B, H] (as parity_util.branch_gradients does for the plain head: two
    correct fp32 implementations may disagree on relu'(z) where z is within round-off of 0)."""
    p = [t.double().requires_grad_(True) for t in params]
    w1, b1, w2, b2, w3, b3, wv, bv = p
    m1, m2 = (torch.as_tensor(np.asarray(m, np.float64)) for m in (mask1, mask2))
    h = torch.baddbmm(b1[:, None, :], torch.as_tensor(states, dtype=torch.float64), w1) * m1
    h = torch.baddbmm(b2[:, None, :], h, w2) * m2
    adv = torch.baddbmm(b3[:, None, :], h, w3)
    q = torch.baddbmm(bv[:, None, :], h, wv) + adv - adv.mean(dim=2, keepdim=True)
    pred = torch.gather(q, 2, torch.as_tensor(actions, dtype=torch.int64)[..., None])[..., 0]
    loss = (pred - torch.as_tensor(y, dtype=torch.float64)).square().mean(dim=1).sum()
    return [g.float() for g in torch.autograd.grad(loss, p)]


@pytest.mark.parametrize("h,precision", [(64, "fp32"), (128, "fp32"), (256, "fp32"), (512, "fp32"), (256, "tf32x3")])
def test_dueling_learn_matches_the_two_stream_oracle(h, precision):
    n, cap, b = 3, 200, 128
    grp = _group(n, cap, b, h=h, precision=precision, **DUEL)
    stk = DuelingStackedOracle(n, 89, [h, h], 4, gamma=0.99, learning_rate=5e-4, target_update_frequency=3, seed0=60)
    rng = np.random.default_rng(h)
    for k in (1, 3, 5, 7):
        stk.online[k] += torch.as_tensor(rng.standard_normal(stk.online[k].shape).astype(np.float32)) * 0.05
        stk.target[k].copy_(stk.online[k])
    _load(grp, stk)
    _fill(grp, [cap + 40, 150, cap], seed=h)
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    # greedy actions against the oracle's, outside near-ties
    x = grp.obs[:, 7].clone()
    acts, q = grp.act(x, return_q=True)
    q_ref = stk.q_values(x[:, :89].cpu().numpy()).numpy()
    close(q.cpu().numpy(), q_ref, what="act Q")
    qs = np.sort(q_ref, axis=1)
    clear = (qs[:, -1] - qs[:, -2]) > RTOL * np.abs(q_ref).max()
    assert np.array_equal(acts.cpu().numpy()[clear], q_ref.argmax(1)[clear])
    for step in range(4):
        metrics = grp.learn(draw_words(rng, n, b)).cpu().numpy()
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        assert int(dbg["tc_error"][0]) == 0
        take = lambda arr, rows: np.stack([arr[g].reshape(-1, *arr.shape[2:])[rows[g] % cap] for g in range(n)])
        S, A_, S2 = take(obs, dbg["rows"]), take(act, dbg["rows"]), take(nobs, dbg["next_rows"])
        th0, m0, v0 = ([p.clone() for p in ps] for ps in (stk.online, stk.adam_m, stk.adam_v))
        t = int(stk.learn_step[0]) + 1
        out = stk.learn_on_batch(S, A_, dbg["r_hat"], S2, None, discounts=dbg["discount"])
        qn = np.sort(out["q_next"], axis=2)
        tie = (qn[..., -1] - qn[..., -2]) < RTOL * np.abs(out["q_next"]).max()
        assert tie.mean() < 0.01
        close(dbg["q_all"], out["q_all"], what=f"step {step} online Q(s)")
        close(dbg["y"][~tie], out["y"][~tie], what=f"step {step} TD target")
        if not tie.any():
            close(metrics[:, 0], out["loss"], what=f"step {step} loss")
            alpha_t, eps_t = adam_scalars(t, 5e-4, "keras")
            g64 = _grads64(th0, S, A_, dbg["y"], dbg["dh1"] != 0, dbg["dh2"] != 0)
            for i in range(n):
                got = [grp.get_weights(i, w) for w in ("online", "m", "v")]
                for k in range(8):
                    gk = g64[k][i]
                    adam_close(got[0][k].numpy(), th0[k][i], m0[k][i], v0[k][i], gk, alpha_t, eps_t,
                               what=f"step {step} net {i} theta[{k}]")
                    close(got[1][k].numpy(), (m0[k][i] + (gk - m0[k][i]) * np.float32(0.1)).numpy(), what=f"m[{k}]")
                    close(got[2][k].numpy(), (v0[k][i] + (gk * gk - v0[k][i]) * np.float32(0.001)).numpy(),
                          rtol=2 * RTOL, what=f"v[{k}]")
        _load(grp, stk)


@pytest.mark.parametrize("tau", [None, 0.05])
def test_free_running_dueling_trajectory_follows_the_oracle(tau):
    n, cap, b, h = 2, 200, 64, 64
    grp = _group(n, cap, b, h=h, tau=tau, normalize_rewards=False, **DUEL)
    stk = DuelingStackedOracle(n, 89, [h, h], 4, gamma=0.99, learning_rate=5e-4, target_update_frequency=3, tau=tau,
                               seed0=70)
    _load(grp, stk)
    _fill(grp, cap, seed=3)
    grp.rew_ring.mul_(1e-3)
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    rng = np.random.default_rng(4)
    for step in range(30):
        metrics = grp.learn(draw_words(rng, n, b)).cpu().numpy()
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        take = lambda arr, rows: np.stack([arr[g][rows[g] % cap] for g in range(n)])
        out = stk.learn_on_batch(take(obs, dbg["rows"]), take(act, dbg["rows"]), dbg["r_hat"], take(nobs, dbg["next_rows"]),
                                 None, discounts=dbg["discount"])
        close(metrics[:, 0], out["loss"], rtol=1e-4, what=f"step {step} loss")
    for i in range(n):
        for which, src in (("online", stk.online), ("target", stk.target)):
            for k, (got, ref) in enumerate(zip(grp.get_weights(i, which), src)):
                close(got.numpy(), ref[i].numpy(), rtol=1e-4, what=f"net {i} {which}[{k}]")


def test_clipping_norm_covers_the_value_head():
    n, cap, b, c = 3, 160, 64, 1e-3
    grp = _group(n, cap, b, h=256, precision="tf32x3", global_clipnorm=c, **DUEL)
    _perturb(grp, 1)
    _fill(grp, cap, seed=5)
    saved = {k: getattr(grp, k).clone() for k in ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step")}
    words = draw_words(np.random.default_rng(6), n, b)
    grp.learn(words)
    end = int(grp.layout.bv) + 4
    g = grp.grads.cpu().numpy()
    assert np.all(g[:, end - 3:] == 0) and np.abs(g[:, grp.layout.wv:grp.layout.bv + 1]).max() > 0
    n64 = np.sqrt((g[:, :end].astype(np.float64) ** 2).sum(axis=1))
    assert ulps(grp.grad_norms.cpu().numpy(), n64.astype(np.float32)).max() <= 1
    after = {k: getattr(grp, k).clone() for k in ("theta", "theta_tgt", "adam_m", "adam_v")}
    for k, t in saved.items():
        getattr(grp, k).copy_(t)
    from dmdqn_b200 import _native as N
    ref = torch.zeros_like(grp.theta)
    _learn_grads(grp, words, ref)
    s = torch.as_tensor(np.array([np.float32(c / max(x, c)) for x in n64], np.float32)).cuda()
    scaled = (ref * s[:, None]).contiguous()
    N.check(grp.lib.dmdqn_adam_apply(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), scaled.data_ptr(),
                                     grp.workspace.data_ptr(), grp.workspace.numel(), _stream()))
    for k, t in after.items():
        assert torch.equal(getattr(grp, k), t), k


@pytest.mark.parametrize("config", [DUEL, dict(DUEL, **PER, **NSTEP)], ids=["uniform", "per_nstep"])
def test_dueling_chained_step_equals_stage_by_stage_step(config):
    chained_step_equals_stage_by_stage_step(config)


@pytest.mark.parametrize("config", [DUEL, dict(DUEL, **PER, **NSTEP)], ids=["uniform", "per_nstep"])
def test_dueling_captured_learn_equals_plain_learn(config):
    captured_learn_equals_plain_learn(config)


def test_dueling_captured_step_host_equals_step_host():
    captured_step_host_equals_step_host(DUEL)


def test_dueling_one_group_of_eight_equals_two_groups_of_four():
    one_group_of_eight_equals_two_groups_of_four(DUEL)


@pytest.mark.parametrize("precision,a", [("fp32", 3), ("tf32x3", 2)])
def test_inactive_networks_and_unused_advantage_columns_stay_untouched(precision, a):
    n, cap, b = 4, 160, 128
    grp = _group(n, cap, b, h=256, precision=precision, a=a, **DUEL)
    _perturb(grp, 2)
    _fill(grp, cap, seed=7)
    L, H = grp.layout, grp.hidden
    mask = torch.tensor([1, 0, 1, 0], dtype=torch.uint8)
    before = {k: getattr(grp, k).clone() for k in ("theta", "theta_tgt", "adam_m", "adam_v")}
    rng = np.random.default_rng(8)
    for _ in range(5):
        grp.learn(draw_words(rng, n, b), mask=mask)
    for k, t in before.items():
        assert torch.equal(getattr(grp, k)[1::2], t[1::2]), k
        w3 = getattr(grp, k)[:, L.w3:L.w3 + 4 * H].view(n, H, 4)
        assert torch.all(w3[..., a:] == 0) and torch.all(getattr(grp, k)[:, L.b3 + a:L.b3 + 4] == 0), k
        assert torch.all(getattr(grp, k)[:, L.bv + 1:] == 0), k
    assert not torch.equal(grp.theta[0, L.wv:L.bv + 1], before["theta"][0, L.wv:L.bv + 1])


@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
def test_dueling_false_equals_a_group_without_the_key(precision):
    n, cap, b = 4, 160, 128
    a, c = _group(n, cap, b, h=256, precision=precision), _group(n, cap, b, h=256, precision=precision, dueling=False)
    for g in (a, c):
        _fill(g, cap, seed=9)
    rng = np.random.default_rng(10)
    for _ in range(4):
        w = draw_words(rng, n, b)
        assert torch.equal(a.learn(w), c.learn(w))
    for k in ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step"):
        assert torch.equal(getattr(a, k), getattr(c, k)), k


@pytest.mark.parametrize("h,precision", [(64, "fp32"), (256, "tf32x3")])
def test_learn_grads_writes_the_whole_adam_range_into_an_uninitialised_buffer(h, precision):
    """The gradient block of a dueling step covers [0, b3 + 8 + H) -- the pad after bv included, as 0 -- whatever the
    buffer held: a NaN-filled buffer gives the block, the clip norm and the clipped update of a zero-filled one."""
    from dmdqn_b200 import _native as N
    n, cap, b, c = 3, 160, 128, 1e-3
    grp = _group(n, cap, b, h=h, precision=precision, **DUEL)
    _perturb(grp, 4)
    _fill(grp, cap, seed=11)
    end = int(grp.layout.bv) + 4
    saved = {k: getattr(grp, k).clone() for k in ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step")}
    words = draw_words(np.random.default_rng(12), n, b)
    out = {}
    for fill in (0.0, float("nan")):
        for k, t in saved.items():
            getattr(grp, k).copy_(t)
        grads = torch.full_like(grp.theta, fill)
        norms = torch.full((n,), fill, device="cuda")
        _learn_grads(grp, words, grads)
        N.check(grp.lib.dmdqn_clip_adam_apply(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), grads.data_ptr(), c,
                                              norms.data_ptr(), grp.workspace.data_ptr(), grp.workspace.numel(), _stream()))
        torch.cuda.synchronize()
        out[fill == 0.0] = (grads[:, :end].clone(), norms.clone(), {k: getattr(grp, k).clone() for k in saved})
    (g0, n0, s0), (g1, n1, s1) = out[True], out[False]
    assert torch.isfinite(g1).all() and torch.all(g1[:, end - 3:] == 0)
    assert torch.equal(g0, g1) and torch.equal(n0, n1) and bool((n1 > c).all())
    for k in s0:
        assert torch.equal(s0[k], s1[k]), k
    assert torch.all(s1["theta"][:, end - 3:] == 0) and torch.all(s1["adam_v"][:, end - 3:] == 0)


# ------------------------------------------------------------------ shared parameters ----------------------------------
def _shared_ranks(world, h, n_agents, b, cap, precision, seed):
    """`world` replicas of one shared dueling network (same weights) with different ring contents."""
    out = []
    for r in range(world):
        grp = _group(n_agents, cap, b, h=h, precision=precision, seed=1, share_parameters=True, target_update_frequency=2,
                     **DUEL)
        _perturb(grp, 9)
        _fill(grp, cap + 2, seed=seed + 17 * r)
        out.append(grp)
    return out


def _fixed_draws(grp, words):
    grp.draw_words = lambda shape, w=words: torch.as_tensor(w.view(np.int32)).to(grp.device)


@pytest.mark.parametrize("h,precision", [(256, "tf32x3"), (64, "fp32")])
def test_dueling_shared_step_world_one_equals_grads_then_adam_apply(h, precision):
    """SharedParameterStep at world 1, on the NCCL path and fused over peer memory, against dmdqn_learn_grads ->
    dmdqn_adam_apply on a twin: the same bits in theta / m / v / theta_tgt (value head included) and the same loss."""
    from dmdqn_b200 import _native as N
    from dmdqn_b200.parallel import PeerExchange, SharedParameterStep
    a, b_, ref = (_shared_ranks(1, h, 3, 64, 60, precision, seed=5)[0] for _ in range(3))
    plain = SharedParameterStep.for_group(a, fused=False)
    fused = SharedParameterStep.for_group(b_, exchange=PeerExchange(b_, 0, 1))
    L = ref.layout
    head0 = ref.theta[0, L.wv:L.bv + 1].clone()
    rng = np.random.default_rng(1)
    for it in range(4):
        words = rng.integers(0, 2**32, (1, 64), dtype=np.uint64).astype(np.uint32)
        for g in (a, b_, ref):
            _fixed_draws(g, words)
        la, lb = plain.step().cpu().numpy(), fused.step().cpu().numpy()
        grads = torch.zeros_like(ref.theta)
        _learn_grads(ref, ref.draw_words((1, 64)), grads)
        N.check(ref.lib.dmdqn_adam_apply(C.byref(ref.dims), C.byref(ref.hp), C.byref(ref.nets), grads.data_ptr(),
                                         ref.workspace.data_ptr(), ref.workspace.numel(), _stream()))
        torch.cuda.synchronize()
        b_.check_errors()
        assert np.array_equal(la.ravel(), lb.ravel()) and np.float32(la.ravel()[0]) == ref.metrics[0, 0].item()
        for name in ("theta", "theta_tgt", "adam_m", "adam_v"):
            assert torch.equal(getattr(a, name), getattr(ref, name)), f"step {it}: NCCL path {name} differs"
            assert torch.equal(getattr(b_, name), getattr(ref, name)), f"step {it}: fused path {name} differs"
    assert not torch.equal(ref.theta[0, L.wv:L.bv + 1], head0)          # the value head learned


@pytest.mark.parametrize("world", [2, 3])
def test_dueling_fused_peer_ranks_match_the_summed_gradient(world):
    """`world` dueling replicas with different rings on one device, each on its own stream: every replica ends
    bit-identical, and equal to twins that apply dmdqn_adam_apply to the rank-ordered sum of the per-rank blocks."""
    from dmdqn_b200 import _native as N
    from dmdqn_b200.parallel import PeerExchange, SharedParameterStep
    h, n_agents, batch, cap = 256, 2, 128, 150
    ranks = _shared_ranks(world, h, n_agents, batch, cap, "tf32x3", seed=40)
    twins = _shared_ranks(world, h, n_agents, batch, cap, "tf32x3", seed=40)
    exchanges = [PeerExchange(g, r, world) for r, g in enumerate(ranks)]
    PeerExchange.connect_local(exchanges)
    steps = [SharedParameterStep.for_group(g, exchange=e) for g, e in zip(ranks, exchanges)]
    streams = [torch.cuda.Stream() for _ in range(world)]
    rng = np.random.default_rng(3)
    for it in range(3):
        words = [rng.integers(0, 2**32, (1, batch), dtype=np.uint64).astype(np.uint32) for _ in range(world)]
        torch.cuda.synchronize()
        losses = []
        for r in range(world):          # gradients first, then the exchange kernels (no rank spins while another learns)
            _fixed_draws(ranks[r], words[r])
            with torch.cuda.stream(streams[r]):
                steps[r].fused_begin(batch * world)
        torch.cuda.synchronize()
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                losses.append(steps[r].fused_finish())
        torch.cuda.synchronize()
        for g in ranks:
            g.check_errors()
        total, loss_sum = None, np.float32(0)
        for r in range(world):
            tw = twins[r]
            gb = torch.zeros_like(tw.theta)
            N.check(tw.lib.dmdqn_learn_grads(C.byref(tw.dims), C.byref(tw.hp), C.byref(tw.replay), C.byref(tw.nets),
                                             torch.as_tensor(words[r].view(np.int32)).cuda().data_ptr(), None, batch * world,
                                             gb.data_ptr(), tw.metrics.data_ptr(), tw.workspace.data_ptr(),
                                             tw.workspace.numel(), _stream()))
            total = gb.clone() if total is None else total + gb
            loss_sum = np.float32(loss_sum + tw.metrics[0, 0].item())
        for tw in twins:
            N.check(tw.lib.dmdqn_adam_apply(C.byref(tw.dims), C.byref(tw.hp), C.byref(tw.nets), total.data_ptr(),
                                            tw.workspace.data_ptr(), tw.workspace.numel(), _stream()))
        torch.cuda.synchronize()
        for r in range(world):
            assert np.float32(losses[r].item()) == loss_sum, f"step {it}: loss of rank {r}"
            for name in ("theta", "theta_tgt", "adam_m", "adam_v"):
                assert torch.equal(getattr(ranks[r], name), getattr(ranks[0], name)), f"step {it}: replica {r} {name}"
                assert torch.equal(getattr(ranks[r], name), getattr(twins[0], name)), f"step {it}: rank {r} {name}"
