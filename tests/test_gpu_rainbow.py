"""Rainbow networks (dueling noisy C51 heads) on the GPU: the noise record, the per-atom fold and projection, the learn step
against dmdqn_learn_grads_dist on the assembled C51 block and against tests/rainbow_oracle.py, Adam, act and the host API."""
import ctypes as C

import numpy as np
import pytest
import torch

import rainbow_oracle as RO
from oracle.dqn import adam_scalars, adam_update_
from parity_util import RTOL, adam_close, close, copy_state, draw_words, fill_rings, ulps

pytestmark = pytest.mark.gpu

STATE = ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step", "metrics", "sigma", "sigma_tgt", "sigma_m", "sigma_v")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def rb_group(n, cap, b, h=64, a=4, atoms=11, seed=0, **extra):
    from dmdqn_b200.group import AgentGroup
    cfg = {"nn_layers": [h, h], "replay_buffer_size": cap, "batch_size": b, "learning_rate": 5e-4, "gamma": 0.99,
           "target_update_frequency": 3, "rainbow": True, "num_atoms": atoms, "v_min": -10.0, "v_max": 10.0}
    cfg.update(extra)
    return AgentGroup(n, cfg, action_size=a, seed=seed)


def dist_twin(grp):
    """A C51 group of the same dims and rings as ``grp`` (its blocks are set by the caller)."""
    from dmdqn_b200.group import AgentGroup
    cfg = dict(grp.config, rainbow=False, distributional=True, precision="fp32")
    c = AgentGroup(grp.n_agents, cfg, action_size=grp.action_size, seed=0)
    for name in ("obs", "next_obs", "act_ring", "rew_ring", "done_ring", "n_written", "priority", "priority_max", "learn_step"):
        if getattr(grp, name) is not None:
            getattr(c, name).copy_(getattr(grp, name))
    c.n_written_host[:] = grp.n_written_host
    return c


def fill(grp, n_written, seed):
    """fill_rings' contents with the observations scaled by 1/8 (the softmax of the heads is not saturated)."""
    fill_rings(grp, n_written, seed=seed, done_rate=0.1)
    grp.act_ring.remainder_(grp.action_size)
    grp.obs.mul_(0.125)
    grp.next_obs.mul_(0.125)


def perturb(grp, seed):
    """Non-zero biases and value weights, a sigma that differs per element and a target that differs from the online
    network; padding stays 0."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    for g in range(grp.n_nets):
        ws = grp.get_weights(g)
        k = len(ws) // 2
        grp.set_weights(g, [w + 0.05 * torch.randn(w.shape, generator=torch.Generator().manual_seed(seed + g)) for w in ws[:k]]
                        + ws[k:], sync_target=True)
    mask = (grp.sigma != 0).float()                 # sigma is 0 exactly on the padding
    grp.theta_tgt.add_(mask * torch.randn(grp.theta.shape, device="cuda", generator=gen) * 0.02)
    for t in (grp.sigma, grp.sigma_tgt):
        t.mul_(0.5 + torch.rand(t.shape, device="cuda", generator=gen))


def keys(grp):
    return [int(k) & ((1 << 64) - 1) for k in grp.key.cpu().tolist()]


def rainbow_fold(grp):
    from dmdqn_b200 import _native as N
    N.check(grp.lib.dmdqn_rainbow_fold(C.byref(grp.dims), C.byref(grp.dist), C.byref(grp.nets), C.byref(grp.noisy_ptrs),
                                       _stream()))


def heads(grp):
    return grp.debug_views()["head"].cpu().numpy()


def assembled(grp, dist_grp, set_):
    """The C51 blocks [n_nets][C51 stride] of eff (set 0) or eff_tgt (1) with the folded heads of the last fold."""
    eff = (grp.eff if set_ == 0 else grp.eff_tgt).cpu().numpy()
    hd = heads(grp)[set_]
    return torch.as_tensor(np.stack([RO.c51_block(eff[g], hd[g], grp.layout, dist_grp.layout.stride)
                                     for g in range(grp.n_nets)])).cuda()


# ------------------------------------------------------------------ 1. noise and fold -------------------------------------
@pytest.mark.parametrize("h,a,atoms", [(64, 4, 11), (128, 3, 2), (256, 2, 51), (64, 4, 64)])
def test_noise_record_eff_and_folded_heads(h, a, atoms):
    grp = rb_group(3, 100, 32, h=h, a=a, atoms=atoms, seed=h + atoms)
    perturb(grp, 5)
    grp.learn_step.copy_(torch.tensor([0, 7, 123], dtype=torch.int32))
    rainbow_fold(grp)
    torch.cuda.synchronize()
    noise, ks = grp.noise.cpu().numpy(), keys(grp)
    for g, t in enumerate((0, 7, 123)):
        for s, (mu, sg, eff) in enumerate(((grp.theta, grp.sigma, grp.eff), (grp.theta_tgt, grp.sigma_tgt, grp.eff_tgt))):
            ref = RO.noise_record(ks[g], t, s, grp.noise_record, 89, a, atoms)
            assert ulps(noise[g, s], ref).max() <= 1, (g, s)
            assert np.array_equal(noise[g, s] == 0, ref == 0)
            e = RO.eps_block(noise[g, s], grp.noise_record, grp.layout, h)
            want = (mu[g].cpu().numpy() + sg[g].cpu().numpy() * e).astype(np.float32)
            assert np.array_equal(eff[g].cpu().numpy(), want), (g, s)
            hd = heads(grp)[s, g]
            assert np.array_equal(hd, RO.fold_heads(eff[g].cpu().numpy(), grp.layout, h, a, atoms)), (g, s)


# ------------------------------------------------------------------ 3. learn step on the assembled block --------------------
def _learn_grads_rainbow(grp, words, grads):
    from dmdqn_b200 import _native as N
    N.check(grp.lib.dmdqn_learn_grads_rainbow(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.dist), C.byref(grp.replay),
                                              C.byref(grp.nets), C.byref(grp.noisy_ptrs), words.data_ptr(), None, grp.batch_size,
                                              grads.data_ptr(), grp.metrics.data_ptr(), grp.workspace.data_ptr(),
                                              grp.workspace.numel(), _stream()))


def _adam_rainbow(grp, grads):
    from dmdqn_b200 import _native as N
    N.check(grp.lib.dmdqn_adam_apply_rainbow(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), C.byref(grp.noisy_ptrs),
                                             grp.num_atoms, grads.data_ptr(), grp.workspace.data_ptr(), grp.workspace.numel(),
                                             _stream()))


@pytest.mark.parametrize("h,a,atoms,extra", [(64, 4, 11, {}), (128, 3, 51, {"sample_mode": "prioritized"}),
                                             (256, 4, 51, {"n_step": 3}), (64, 2, 2, {"double_dqn": False}),
                                             (512, 3, 64, {})])
def test_learn_grads_equal_the_dist_call_on_the_assembled_block(h, a, atoms, extra):
    from dmdqn_b200 import _native as N
    n, cap, b = 3, 200, 64
    grp = rb_group(n, cap, b, h=h, a=a, atoms=atoms, seed=h, **extra)
    perturb(grp, h)
    fill(grp, [cap + 40, 150, cap], seed=h + atoms)
    grp.learn_step.fill_(4)
    c = dist_twin(grp)
    rainbow_fold(grp)
    c.theta.copy_(assembled(grp, c, 0))
    c.theta_tgt.copy_(assembled(grp, c, 1))
    w = draw_words(np.random.default_rng(h), n, b)
    grads = torch.zeros_like(grp.theta)
    _learn_grads_rainbow(grp, w, grads)
    gd = torch.zeros_like(c.theta)
    N.check(c.lib.dmdqn_learn_grads_dist(C.byref(c.dims), C.byref(c.hp), C.byref(c.dist), C.byref(c.replay), C.byref(c.nets),
                                         w.data_ptr(), None, b, gd.data_ptr(), c.metrics.data_ptr(), c.workspace.data_ptr(),
                                         c.workspace.numel(), None))
    torch.cuda.synchronize()
    assert torch.equal(grp.metrics, c.metrics)
    dr, dd = grp.debug_views(), c.debug_views()
    for k in ("q_all", "q_next", "tq_all", "rows", "next_rows", "target_dist", "dlogits", "h2", "dh1", "dh2"):
        assert torch.equal(dr[k], dd[k]), k
    if grp.prioritized:
        assert torch.equal(grp.priority, c.priority) and torch.equal(grp.priority_max, c.priority_max)
    L = grp.layout
    gd_np, gr_np = gd.cpu().numpy(), grads.cpu().numpy()
    for g in range(n):
        assert np.array_equal(gr_np[g, :L.w3], gd_np[g, :L.w3]), g
        full = np.zeros(int(L.stride), np.float32)
        full[:L.wv] = gd_np[g, :L.wv]
        want = RO.project_heads(full, L, h, a, atoms)
        assert np.array_equal(gr_np[g, :L.end], want[:L.end]), g


# ------------------------------------------------------------------ 4. Adam ---------------------------------------------------
@pytest.mark.parametrize("tau", [None, 0.05])
def test_adam_is_adam_on_mu_with_g_and_on_sigma_with_g_times_eps(tau):
    n, cap, b, h = 2, 200, 64, 64
    grp = rb_group(n, cap, b, h=h, tau=tau, seed=3)
    perturb(grp, 3)
    fill(grp, cap, seed=4)
    grp.learn_step.fill_(2)             # hard sync at step 3
    before = {k: getattr(grp, k).clone() for k in STATE}
    grads = torch.zeros_like(grp.theta)
    _learn_grads_rainbow(grp, draw_words(np.random.default_rng(1), n, b), grads)
    _adam_rainbow(grp, grads)
    torch.cuda.synchronize()
    L, alpha, eps = grp.layout, *adam_scalars(3, 5e-4, "keras")
    for g in range(n):
        e = torch.as_tensor(RO.eps_block(grp.noise[g, 0].cpu().numpy(), grp.noise_record, L, h))
        gg = grads[g].cpu()
        for p, m, v, tg, gr in (("theta", "adam_m", "adam_v", "theta_tgt", gg), ("sigma", "sigma_m", "sigma_v", "sigma_tgt", gg * e)):
            th, mm, vv = (before[k][g].cpu().clone() for k in (p, m, v))
            th, mm, vv, gr = th[:L.end], mm[:L.end], vv[:L.end], gr[:L.end]
            adam_update_(th, gr, mm, vv, alpha, eps)
            close(getattr(grp, p)[g, :L.end].cpu().numpy(), th.numpy(), what=p)
            close(getattr(grp, m)[g, :L.end].cpu().numpy(), mm.numpy(), what=m)
            close(getattr(grp, v)[g, :L.end].cpu().numpy(), vv.numpy(), rtol=2 * RTOL, what=v)
            if tau is None:
                assert torch.equal(getattr(grp, tg)[g], getattr(grp, p)[g]), tg
            else:
                t32 = float(np.float32(tau))
                close(getattr(grp, tg)[g].cpu().numpy(),
                      (t32 * getattr(grp, p)[g] + (1.0 - t32) * before[tg][g]).cpu().numpy(), what=tg)
        assert torch.equal(grp.theta[g, L.end:], before["theta"][g, L.end:])


# ------------------------------------------------------------------ 5. against the oracle -------------------------------------
def oracle_for(grp, **kw):
    stk = RO.RainbowOracle(grp.n_nets, 89, [grp.hidden] * 2, grp.action_size, grp.num_atoms, -10.0, 10.0, gamma=0.99,
                           learning_rate=5e-4, target_update_frequency=3, **kw)
    lists = []
    for which in ("online", "target", "m", "v"):
        per = [grp.get_weights(i, which) for i in range(grp.n_nets)]
        k = len(per[0]) // 2
        lists.append(([torch.stack([p[j] for p in per]) for j in range(k)], [torch.stack([p[k + j] for p in per]) for j in range(k)]))
    (mu, sg), (mt, st), (m, sm), (v, sv) = lists
    stk.set_state(mu, sg, mt, st, m, v, sm, sv)
    stk.learn_step[:] = grp.learn_step.cpu().numpy()
    return stk


def step_eps(grp, s):
    noise = grp.noise.cpu().numpy()
    per = [RO.eps_params(noise[g, s], grp.noise_record, 89, grp.action_size, grp.num_atoms) for g in range(grp.n_nets)]
    return [torch.stack([p[k] for p in per]) for k in range(len(per[0]))]


def oracle_step(grp, stk, rng):
    cap = grp.capacity
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    metrics = grp.learn(draw_words(rng, grp.n_nets, grp.batch_size)).cpu().numpy()
    dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
    take = lambda arr, rows: np.stack([arr[g][rows[g] % cap] for g in range(grp.n_nets)])
    out = stk.learn_on_batch(take(obs, dbg["rows"]), take(act, dbg["rows"]), dbg["r_hat"], take(nobs, dbg["next_rows"]), None,
                             step_eps(grp, 0), step_eps(grp, 1), discounts=dbg["discount"],
                             is_weights=dbg["is_weights"] if grp.prioritized else None)
    return metrics, dbg, out


def one_step(h, a, atoms, **extra):
    n, cap, b = 3, 200, 64
    grp = rb_group(n, cap, b, h=h, a=a, atoms=atoms, seed=h + a, **extra)
    perturb(grp, h + atoms)
    fill(grp, [cap + 40, 150, cap], seed=h + atoms)
    stk = oracle_for(grp, double_dqn=extra.get("double_dqn", True))
    th0 = [[p.clone() for p in ps] for ps in (stk.online, stk.adam_m, stk.adam_v, stk.sigma, stk.sigma_m, stk.sigma_v)]
    t = int(stk.learn_step[0]) + 1
    metrics, dbg, out = oracle_step(grp, stk, np.random.default_rng(h + atoms))
    for key in ("q_all", "q_next", "tq_all"):
        close(dbg[key][..., :a], out[key], what=key)
    sel = np.sort(out["q_next"] if extra.get("double_dqn", True) else out["tq_all"], axis=2)
    tie = (sel[..., -1] - sel[..., -2]) < 4 * RTOL * np.abs(sel).max() if a > 1 else np.zeros(sel.shape[:2], bool)
    close(dbg["target_dist"][..., :atoms][~tie], out["m"][~tie], scale=1.0, what="projected distribution")
    alpha_t, eps_t = adam_scalars(t, 5e-4, "keras")
    for i in range(n):
        if tie[i].any():
            continue
        close(metrics[i, 0], out["loss"][i], what=f"net {i} loss")
        got = grp.get_weights(i, "online")
        k = len(got) // 2
        for j in range(2 * k):
            ps, ms, vs = (th0[0], th0[1], th0[2]) if j < k else (th0[3], th0[4], th0[5])
            gk = torch.as_tensor((out["g_mu"] if j < k else out["g_sigma"])[j % k][i])
            adam_close(got[j].numpy(), ps[j % k][i], ms[j % k][i], vs[j % k][i], gk, alpha_t, eps_t, what=f"net {i} param {j}")


@pytest.mark.parametrize("h,a,atoms", [(64, 2, 2), (64, 4, 51), (128, 3, 64), (256, 4, 51), (512, 3, 11)])
def test_one_step_matches_the_oracle(h, a, atoms):
    one_step(h, a, atoms)


@pytest.mark.parametrize("extra", [{"sample_mode": "prioritized"}, {"n_step": 3}, {"double_dqn": False}])
def test_learn_variants_match_the_oracle(extra):
    one_step(64, 4, 11, **extra)


def test_free_running_trajectory_follows_the_oracle():
    n, cap, b, h = 2, 200, 64, 64
    grp = rb_group(n, cap, b, h=h, a=4, atoms=11, normalize_rewards=False, seed=1)
    fill(grp, cap, seed=3)
    grp.rew_ring.mul_(1e-2)
    stk = oracle_for(grp)
    rng = np.random.default_rng(4)
    for step in range(30):
        metrics, _, out = oracle_step(grp, stk, rng)
        close(metrics[:, 0], out["loss"], rtol=1e-4, what=f"step {step} loss")
    for i in range(n):
        for which, mu, sg in (("online", stk.online, stk.sigma), ("target", stk.target, stk.sigma_tgt)):
            got = grp.get_weights(i, which)
            for j, ref in enumerate(mu + sg):
                close(got[j].numpy(), ref[i].numpy(), rtol=1e-4, what=f"{which} {j}")


# ------------------------------------------------------------------ 6. act ------------------------------------------------------
def _act_inputs(n, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    obs = torch.randn((n, 96), device="cuda", generator=gen) * 0.5
    obs[:, 89:] = 0
    eps = np.where(np.arange(n) % 4 == 3, 1.0, 0.0)              # agents 3, 7, ... explore
    return obs, eps, np.zeros(n, np.uint32), (np.arange(n, dtype=np.uint64) * 0x40000000).astype(np.uint32)


def _same_act(x, y):
    (ax, qx), (ay, qy) = x, y
    assert torch.equal(ax, ay)
    assert torch.equal(torch.isnan(qx), torch.isnan(qy)) and torch.equal(torch.nan_to_num(qx), torch.nan_to_num(qy))


@pytest.mark.parametrize("h,a,atoms", [(64, 4, 11), (128, 3, 51), (256, 4, 51), (512, 2, 64)])
def test_act_equals_act_dist_on_the_assembled_block(h, a, atoms):
    n = 8
    grp = rb_group(n, 100, 32, h=h, a=a, atoms=atoms, seed=h)
    perturb(grp, h)
    grp.learn_step.copy_(torch.arange(n, dtype=torch.int32) * 3)
    c = dist_twin(grp)
    obs, eps, we, wa = _act_inputs(n, h)
    rainbow_fold(grp)                                               # noisy: eff's trunk and its folded head
    c.theta.copy_(assembled(grp, c, 0))
    got = grp.act(obs, eps, we, wa, return_q=True)
    _same_act(got, c.act(obs, eps, we, wa, return_q=True))
    assert torch.isnan(got[1][3]).all() and not torch.isnan(got[1][0]).any()
    mu = grp.theta.cpu().numpy()                                    # greedy: mu, the fold restated on the CPU
    c.theta.copy_(torch.as_tensor(np.stack([RO.c51_block(mu[g], RO.fold_heads(mu[g], grp.layout, h, a, atoms), grp.layout,
                                                         c.layout.stride) for g in range(n)])).cuda())
    _same_act(grp.act(obs, eps, we, wa, return_q=True, noisy=False), c.act(obs, eps, we, wa, return_q=True))


def test_act_after_a_learn_step_uses_the_next_steps_online_noise():
    grp = rb_group(4, 200, 64, seed=2)
    perturb(grp, 2)
    fill(grp, 200, seed=2)
    grp.learn(draw_words(np.random.default_rng(2), 4, 64))
    obs, eps, we, wa = _act_inputs(4, 2)
    got = grp.act(obs, eps, we, wa, return_q=True)
    rainbow_fold(grp)                                               # at the advanced learn_step
    c = dist_twin(grp)
    c.theta.copy_(assembled(grp, c, 0))
    _same_act(got, c.act(obs, eps, we, wa, return_q=True))


# ------------------------------------------------------------------ 7. call patterns ---------------------------------------------
def _twins(n=6, cap=200, b=64, **extra):
    a, c = (rb_group(n, cap, b, h=128, seed=7, **extra) for _ in range(2))
    for g in (a, c):
        fill(g, cap, seed=8)
    return a, c


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
        for name in STATE + ("noise",) + (("priority",) if a.prioritized else ()):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name}"


def test_captured_step_host_equals_step_host():
    n, b = 6, 64
    a, c = _twins(n=n, b=b)
    sa, sc = a.make_step_block(), c.make_step_block()
    rng = np.random.default_rng(13)
    replay = None
    for it in range(4):
        vals = {"obs": rng.integers(-1, 3, (n, 89)).astype(np.float32), "next_obs": rng.integers(-1, 3, (n, 89)).astype(np.float32),
                "act": rng.integers(0, 4, n).astype(np.int32), "rew": -rng.random(n) * 10,
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


def test_inactive_networks_keep_every_tensor():
    grp = rb_group(4, 200, 64, seed=6)
    perturb(grp, 6)
    fill(grp, [200, 10, 200, 200], seed=7)                 # network 1 holds fewer than batch transitions
    before = {k: getattr(grp, k).clone() for k in STATE if k != "metrics"}
    m = grp.learn(draw_words(np.random.default_rng(8), 4, 64), mask=np.array([1, 1, 1, 0], np.uint8)).cpu().numpy()
    assert list(m[:, 7]) == [1, 0, 1, 0] and np.all(m[[1, 3]] == 0)
    for k, v in before.items():
        for g in (1, 3):
            assert torch.equal(getattr(grp, k)[g], v[g]), (k, g)
        assert not torch.equal(getattr(grp, k)[0], v[0]) or k in ("theta_tgt", "sigma_tgt"), k


def test_one_group_of_eight_equals_two_groups_of_four():
    n, cap, b = 8, 300, 64
    big = rb_group(n, cap, b, h=128, seed=14)
    perturb(big, 14)
    fill(big, [cap + 5, cap, 250, 400, 300, 129, 1000, 301], seed=15)
    halves = [rb_group(4, cap, b, h=128, seed=99) for _ in range(2)]
    for k, hg in enumerate(halves):
        sl = slice(4 * k, 4 * k + 4)
        copy_state(hg, big, sl)
        for name in ("sigma", "sigma_tgt", "sigma_m", "sigma_v", "key"):
            getattr(hg, name).copy_(getattr(big, name)[sl])
    rng = np.random.default_rng(16)
    for it in range(3):
        w = draw_words(rng, n, b)
        mb = big.learn(w).clone()
        mh = torch.cat([hg.learn(w[4 * k:4 * k + 4].contiguous()).clone() for k, hg in enumerate(halves)])
        torch.cuda.synchronize()
        assert torch.equal(mb, mh), it
        for name in STATE + ("noise",):
            assert torch.equal(getattr(big, name), torch.cat([getattr(hg, name) for hg in halves])), (it, name)


# ------------------------------------------------------------------ 8. shared parameters -----------------------------------------
def test_shared_step_world_one_equals_learn_grads_plus_adam():
    from dmdqn_b200.parallel import SharedParameterStep
    n, cap, b = 4, 200, 64
    a, c = (rb_group(n, cap, b, share_parameters=True, seed=3) for _ in range(2))
    for g in (a, c):
        fill(g, cap, seed=3)
    step = SharedParameterStep.for_group(a)
    assert step.fused_apply is None
    with pytest.raises(ValueError, match="rainbow"):
        SharedParameterStep.for_group(a, fused=True)
    for it in range(3):
        a._gen.manual_seed(100 + it); c._gen.manual_seed(100 + it)
        step.step()
        grads = torch.zeros_like(c.theta)
        _learn_grads_rainbow(c, c.draw_words((1, b)), grads)
        _adam_rainbow(c, grads)
        c.learn_step_host += 1
        torch.cuda.synchronize()
        for k in STATE:
            assert torch.equal(getattr(a, k), getattr(c, k)), (it, k)


@pytest.mark.parametrize("world", [2, 3])
def test_simulated_ranks_stay_bit_identical(world):
    n, cap, b = 2, 200, 64
    ranks = [rb_group(n, cap, b, share_parameters=True, seed=1) for _ in range(world)]
    for r, g in enumerate(ranks):
        fill(g, cap, seed=20 + r)
    for it in range(2):
        blocks = []
        for g in ranks:
            grads = torch.zeros_like(g.theta)
            _learn_grads_rainbow(g, g.draw_words((1, b)), grads)
            blocks.append(grads)
        total = blocks[0].clone()
        for blk in blocks[1:]:
            total += blk
        for g in ranks:
            assert torch.equal(g.noise, ranks[0].noise)
            _adam_rainbow(g, total)
        torch.cuda.synchronize()
        for g in ranks[1:]:
            for k in STATE:
                if k != "metrics":
                    assert torch.equal(getattr(g, k), getattr(ranks[0], k)), (it, k)


# ------------------------------------------------------------------ 9. weights and the train loop --------------------------------
def test_weights_round_trip_and_w1_to_b3_are_a_c51_groups_init(tmp_path):
    from dmdqn_b200.agent import DQNAgent
    grp = rb_group(2, 100, 32, h=64, a=3, atoms=11, seed=5)
    c51 = dist_twin(grp)
    c51.init_weights(5)
    ws = grp.get_weights(1)
    shapes = [(89, 64), (64,), (64, 64), (64,), (64, 33), (33,), (64, 11), (11,)]
    assert [tuple(w.shape) for w in ws] == shapes * 2
    for x, y in zip(ws[:6], c51.get_weights(1)):
        assert torch.equal(x, y)
    assert ws[6].abs().max() > 0 and torch.all(ws[7] == 0)
    new = [w + 0.25 for w in ws]
    grp.set_weights(0, new, sync_target=True)
    for x, y in zip(grp.get_weights(0), new):
        assert torch.equal(x, y)
    assert torch.equal(grp.theta[0], grp.theta_tgt[0]) and torch.equal(grp.sigma[0], grp.sigma_tgt[0])
    L, npad = grp.layout, grp.atom_stride
    assert not torch.any(grp.theta[:, L.wv:L.bv].view(2, 64, npad)[:, :, 11:] != 0)
    cfg = {"nn_layers": [64, 64], "replay_buffer_size": 100, "batch_size": 32, "rainbow": True, "num_atoms": 11}
    ag = DQNAgent(89, 3, "a0", cfg)
    assert ag.get_epsilon() == 0
    ag._g.set_weights(0, new)
    path = str(tmp_path / "m.pt")
    ag.save_model(path)
    other = DQNAgent(89, 3, "a1", cfg)
    assert other.load_model(path)
    for x, y in zip(other._g.get_weights(0), new):
        assert torch.equal(x, y)


def test_train_loop_runs_rainbow_from_the_config():
    from dmdqn_b200.train import PRESETS, train_agents
    cfg = dict(PRESETS["shipped_train_py"])
    cfg.update(max_sim_time=600.0, backend="fake", grid_rows=3, grid_cols=3, fake_traci_seed=11, batch_size=16,
               nn_layers=[64, 64], precision="auto", rainbow=True, num_atoms=51, sample_mode="prioritized", n_step=3)
    history, agents, group = train_agents(cfg, episodes=1, mode="batched", seed=3, learn=True)
    t = len(history)
    assert group.rainbow and group.noisy and group.hp.precision == 0 and group.hp.dueling == 1
    assert t > 16 and np.all(group.learn_step.cpu().numpy() == t - 15)
    losses = [h["total_loss"] for h in history]
    assert np.all(np.isfinite(losses)) and any(x != 0 for x in losses)
