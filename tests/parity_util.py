"""Tolerance helpers shared by the GPU parity tests, and the ring fixtures and test bodies that the prioritized-replay
(tests/test_gpu_prioritized.py) and n-step (tests/test_gpu_nstep.py) GPU tests share."""
import ctypes as C

import numpy as np
import torch

import replay_oracle as O
from oracle import replay as R
from oracle.replay import RingReplay

RTOL = 1e-5   # BASELINE.json: "within 1e-5 relative for fp32 Q-values, losses and post-Adam weights"


def close(got, ref, rtol=RTOL, scale=None, what=""):
    """|got-ref| <= rtol * max(|ref| elementwise, magnitude of the tensor)."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    mag = float(np.abs(ref).max()) if scale is None else scale
    tol = rtol * np.maximum(np.abs(ref), mag if mag > 0 else 1.0)
    bad = np.abs(got - ref) > tol
    assert not bad.any(), f"{what}: {bad.sum()} / {bad.size} off, worst {np.abs(got - ref).max():.3e} (mag {mag:.3e})"


def adam_close(got, theta0, m0, v0, grad, alpha, eps, rtol=RTOL, what=""):
    """Post-Adam weights against the oracle, honouring Adam's conditioning.

    Adam divides by sqrt(v): where a gradient element is within round-off of zero the step
    (|step| <= ~lr) is not determined by the inputs to 1e-5 -- the quotient g/(|g|+eps') is.
    So the oracle update is evaluated at g and g +- delta with delta = rtol * max|g| (what
    "gradients equal to 1e-5 relative" means for this tensor) and the kernel's weight must
    lie in that interval, widened by rtol * max(|theta|, max|theta|)."""
    from oracle.dqn import adam_update_
    g = torch.as_tensor(grad)
    delta = rtol * float(g.abs().max())
    cands = []
    for s in (-1.0, 0.0, 1.0):
        p, m, v = theta0.clone(), m0.clone(), v0.clone()
        adam_update_(p, g + s * delta, m, v, alpha, eps)
        cands.append(p.numpy().astype(np.float64))
    lo, hi = np.minimum.reduce(cands), np.maximum.reduce(cands)
    ref = cands[1]
    got = np.asarray(got, np.float64)
    tol = rtol * np.maximum(np.abs(ref), float(np.abs(ref).max()))
    bad = (got < lo - tol) | (got > hi + tol)
    loose = np.abs(got - ref) > tol
    assert not bad.any(), f"{what}: {bad.sum()} / {bad.size} outside the Adam interval, worst {np.abs(got - ref).max():.3e}"
    # the ill-conditioned elements must stay a vanishing minority
    # (a floor of 3 elements: on a 256-element bias vector one ill-conditioned element is already 0.4 %)
    assert loose.sum() <= max(3, 1e-3 * loose.size), f"{what}: {loose.sum()} / {loose.size} elements needed the gradient-interval allowance"
    return int(loose.sum())


def branch_gradients(params, states, actions, y, loss_kind, mask1, mask2, rtol=RTOL, weights=None):
    """Exact (float64) gradients of the batch-mean loss (``weights[N,B]``: of mean_i(w_i * term_i),
    the importance-weighted loss; None = 1) on the piecewise-linear branch the kernel
    took: relu' masks ``mask1``/``mask2`` [N,B,H] come from the kernel's own dh1/dh2 (non-zero
    pattern).  Two correct fp32 implementations may disagree on relu'(z) when z is within
    round-off of 0; this makes that choice an input instead of loosening the tolerance, and
    asserts the masks differ from the oracle's only at such kinks.  SURVEY.md App. A.8 formulas."""
    w1, b1, w2, b2, w3, b3 = (np.asarray(p, np.float64) for p in params)
    x = np.asarray(states, np.float64)
    n, b, _ = x.shape
    z1 = np.einsum("nbd,ndh->nbh", x, w1) + b1[:, None, :]
    h1 = np.maximum(z1, 0)
    z2 = np.einsum("nbh,nhk->nbk", h1, w2) + b2[:, None, :]
    h2 = np.maximum(z2, 0)
    q = np.einsum("nbh,nha->nba", h2, w3) + b3[:, None, :]
    a = np.asarray(actions, np.int64)
    pred = np.take_along_axis(q, a[..., None], 2)[..., 0]
    e = pred - np.asarray(y, np.float64)
    gcoef = 2 * e / b if loss_kind == "mse" else np.clip(e, -1, 1) / b
    if weights is not None:
        gcoef = gcoef * np.asarray(weights, np.float64)
    dq = np.zeros_like(q)
    np.put_along_axis(dq, a[..., None], gcoef[..., None], 2)
    m1 = np.asarray(mask1, bool)
    m2 = np.asarray(mask2, bool)
    for z, m, name in ((z1, m1, "layer 1"), (z2, m2, "layer 2")):
        kink = np.abs(z) < 4 * rtol * np.abs(z).max()
        # the kernel may only treat a unit as active away from the kink if it is active (a unit it
        # treats as inactive although z > 0 shows up as a gradient mismatch below, unless dq W3^T == 0)
        assert not (m & (z <= 0) & ~kink).any(), f"{name}: relu mask set where the pre-activation is clearly negative"
    dh2_all = np.einsum("nba,nha->nbh", dq, w3)
    dh2 = dh2_all * m2
    dh1 = np.einsum("nbk,nhk->nbh", dh2, w2) * m1
    grads = [np.einsum("nbd,nbh->ndh", x, dh1), dh1.sum(1), np.einsum("nbh,nbk->nhk", h1, dh2), dh2.sum(1),
             np.einsum("nbh,nba->nha", h2, dq), dq.sum(1)]
    return [g.astype(np.float32) for g in grads]


def relu_boundary(params, states, rtol=RTOL):
    """Units whose pre-activation sits within round-off of the ReLU kink for some sampled row.

    relu'(z) flips there between two correct fp32 implementations (different summation order),
    which changes one whole column of that layer's weight gradient.  Returns (cols1[N] list of
    sets, hit2[N] bools): layer-1 columns to leave out of the W1/b1 comparison, and whether a
    layer-2 unit is affected (then the gradients of every earlier tensor move too and the
    network is skipped for that step).  float64 evaluation of the oracle's weights."""
    w1, b1, w2, b2 = (np.asarray(p, np.float64) for p in params[:4])
    x = np.asarray(states, np.float64)
    z1 = np.einsum("nbd,ndh->nbh", x, w1) + b1[:, None, :]
    z2 = np.einsum("nbh,nhk->nbk", np.maximum(z1, 0), w2) + b2[:, None, :]
    cols1, hit2 = [], []
    for i in range(x.shape[0]):
        near1 = np.abs(z1[i]) < 4 * rtol * np.abs(z1[i]).max()
        cols1.append(set(np.nonzero(near1.any(axis=0))[0].tolist()))
        hit2.append(bool((np.abs(z2[i]) < 4 * rtol * np.abs(z2[i]).max()).any()))
    return cols1, hit2


def drop_cols(got, ref, cols):
    """Copy of ``got`` with the given last-axis columns replaced by the reference's."""
    if not cols:
        return got
    out = np.array(got, copy=True)
    idx = sorted(cols)
    out[..., idx] = np.asarray(ref)[..., idx]
    return out


# ------------------------------------------------------------------ replay fixtures (prioritized replay, n-step) --------
PER = {"sample_mode": "prioritized"}
NSTEP = {"n_step": 3}


def replay_group(n, cap, b, h=64, precision="fp32", seed=0, **extra):
    from dmdqn_b200.group import AgentGroup
    cfg = {"nn_layers": [h, h], "replay_buffer_size": cap, "batch_size": b, "learning_rate": 5e-4, "gamma": 0.99,
           "target_update_frequency": 3, "precision": precision}
    cfg.update(extra)
    return AgentGroup(n, cfg, seed=seed)


def fill_rings(grp, n_written, seed, done_rate=0.05, priorities=True):
    """Ring contents straight into the device tensors; n_written per agent; non-integer priorities on the written slots."""
    n, cap = grp.n_agents, grp.capacity
    gen = torch.Generator(device="cuda").manual_seed(seed)
    grp.obs[:, :, :89] = torch.randint(-1, 20, (n, cap, 89), device="cuda", generator=gen).float()
    grp.next_obs[:, :, :89] = torch.randint(-1, 20, (n, cap, 89), device="cuda", generator=gen).float()
    grp.act_ring.copy_(torch.randint(0, 4, (n, cap), device="cuda", generator=gen).int())
    grp.rew_ring.copy_(-torch.randint(0, 5000, (n, cap), device="cuda", generator=gen).double() * 0.7)
    grp.done_ring.copy_((torch.rand((n, cap), device="cuda", generator=gen) < done_rate).to(torch.uint8))
    nw = np.broadcast_to(np.asarray(n_written, np.int64), (n,)).copy()
    grp.n_written.copy_(torch.as_tensor(nw)); grp.n_written_host[:] = nw
    if priorities and grp.priority is not None:
        size = torch.as_tensor(np.minimum(nw, cap), device="cuda")
        written = torch.arange(cap, device="cuda")[None, :] < size[:, None]
        p = torch.rand((n, cap), device="cuda", generator=gen) * 2 + 0.01
        grp.priority.copy_(torch.where(written, p, torch.zeros_like(p)))
        grp.priority_max.copy_(grp.priority.max(1).values)


def host_ring(grp):
    """The group's rewards, done flags and fill levels as an oracle ring (observations are compared separately)."""
    ring = RingReplay(grp.n_agents, grp.capacity, 1)
    ring.rew = grp.rew_ring.cpu().numpy()
    ring.done = grp.done_ring.cpu().numpy()
    ring.n_written = grp.n_written.cpu().numpy().astype(np.int64)
    return ring


def draw_words(rng, n, b):
    return torch.as_tensor(rng.integers(0, 2**32, (n, b), dtype=np.uint64).astype(np.uint32).view(np.int32)).cuda()


def ulps(a, b):
    return np.abs(np.asarray(a, np.float32).view(np.int32).astype(np.int64) - np.asarray(b, np.float32).view(np.int32))


def copy_state(dst, src, sl=slice(None)):
    for name in ("obs", "next_obs", "act_ring", "rew_ring", "done_ring", "n_written", "priority", "priority_max",
                 "theta", "theta_tgt", "adam_m", "adam_v", "learn_step"):
        if getattr(src, name) is not None:
            getattr(dst, name).copy_(getattr(src, name)[sl])
    dst.n_written_host[:] = src.n_written_host[sl]
    dst.learn_step_host[:] = src.learn_step_host[sl]


def state_names(grp, *extra):
    """The learned state, the ring's priorities where the group has them, and ``extra``."""
    names = ["theta", "theta_tgt", "adam_m", "adam_v"] + (["priority", "priority_max"] if grp.prioritized else [])
    return names + list(extra)


def check_nstep_against_oracle(grp, ring, dbg, n, normalize=True, what=""):
    """rows -> the oracle's returns, discounts, terminal flags and bootstrap rows, bit for bit; returns the oracle per net."""
    cap, outs = grp.capacity, []
    for g in range(grp.n_nets):
        rows = dbg["rows"][g]
        out = O.nstep_batch(ring, rows // cap, rows % cap, n, 0.99, normalize)
        assert np.array_equal(dbg["next_rows"][g], (rows // cap) * cap + out["next_slot"]), f"{what} net {g}: bootstrap rows"
        assert np.array_equal(dbg["r_hat"][g], out["r_hat"]), f"{what} net {g}: returns"
        assert np.array_equal(dbg["discount"][g], out["discount"]), f"{what} net {g}: discounts"
        outs.append(out)
    return outs


# ------------------------------------------------------------------ shared test bodies ----------------------------------
def learn_matches_the_oracle(h, precision, loss, double_dqn, mode, n_step):
    """Drawn slots, importance weights while beta anneals, returns, discounts, Q, TD targets, the (weighted) loss and the
    Adam step, and the new priorities of the drawn slots."""
    from oracle.dqn import adam_scalars
    n, cap, b, alpha, eps, beta0, beta_steps = 3, 200, 128, 0.6, 1e-6, 0.4, 4
    prioritized = mode == "prioritized"
    grp = replay_group(n, cap, b, h=h, precision=precision, loss=loss, double_dqn=double_dqn, sample_mode=mode, n_step=n_step,
                 per_alpha=alpha, per_eps=eps, per_beta=beta0, per_beta_steps=beta_steps)
    rng = np.random.default_rng(h + len(loss) + double_dqn)
    stk = O.ReplayStackedOracle(n, 89, [h, h], 4, gamma=0.99, learning_rate=5e-4, loss=loss, target_update_frequency=3,
                                double_dqn=double_dqn, seed0=50)
    for k in (1, 3, 5):
        stk.online[k] += torch.as_tensor(rng.standard_normal(stk.online[k].shape).astype(np.float32)) * 0.05
        stk.target[k].copy_(stk.online[k])

    def load():
        for i in range(n):
            for which, src in (("online", stk.online), ("target", stk.target), ("m", stk.adam_m), ("v", stk.adam_v)):
                grp.set_weights(i, [p[i] for p in src], which)
    load()
    fill_rings(grp, [cap + 40, 150, cap], seed=h, done_rate=0.1)
    ring = host_ring(grp)
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    rew = grp.rew_ring.cpu().numpy()
    for step in range(6):
        words = draw_words(rng, n, b)
        if prioritized:
            pr0, pmax0 = grp.priority.cpu().numpy(), grp.priority_max.cpu().numpy()
        metrics = grp.learn(words).cpu().numpy()
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        assert int(dbg["tc_error"][0]) == 0
        t = int(stk.learn_step[0]) + 1
        slots, nslots = dbg["rows"] % cap, dbg["next_rows"] % cap
        isw = None
        if prioritized:
            w = words.cpu().numpy().view(np.uint32)
            beta = O.beta_schedule(t, beta0, beta_steps)
            for g in range(n):
                assert np.array_equal(slots[g], O.prioritized_indices(pr0[g], w[g])), f"step {step} agent {g}: slots"
                assert ulps(dbg["is_weights"][g], O.is_weights(pr0[g], slots[g], beta)).max() <= 2
            isw = dbg["is_weights"]
        outs = check_nstep_against_oracle(grp, ring, dbg, n_step, what=f"step {step}")
        if n_step == 1:
            Rw = np.stack([R.zscore_canonical(rew[g, slots[g]]) for g in range(n)]).astype(np.float32)
            assert np.array_equal(dbg["r_hat"], Rw)
        take = lambda a, s: np.stack([a[g, s[g]] for g in range(n)])
        S, A_, S2 = take(obs, slots), take(act, slots), take(nobs, nslots)
        Rn, D, disc = (np.stack([o[k] for o in outs]) for k in ("r_hat", "done", "discount"))
        th0 = [p.clone() for p in stk.online]; m0 = [p.clone() for p in stk.adam_m]; v0 = [p.clone() for p in stk.adam_v]
        out = stk.learn_on_batch(S, A_, Rn, S2, D, is_weights=isw, discounts=disc)
        qn = np.sort(out["q_next"], axis=2)
        tie = (qn[..., -1] - qn[..., -2]) < RTOL * np.abs(out["q_next"]).max()
        assert tie.mean() < 0.01
        close(dbg["q_all"], out["q_all"], what=f"step {step} online Q(s)")
        close(dbg["y"][~tie], out["y"][~tie], what=f"step {step} TD target")
        if prioritized:                                # the new priorities come from the device's own q(s)[a] and y, within
            delta = np.take_along_axis(dbg["q_all"], A_[..., None].astype(np.int64), 2)[..., 0] - dbg["y"]   # 1 ulp
            pr1, pmax1 = grp.priority.cpu().numpy(), grp.priority_max.cpu().numpy()
            for g in range(n):
                pref = O.priority_of(delta[g], alpha, eps)
                assert ulps(pr1[g, slots[g]], pref).max() <= 1, f"step {step} agent {g}: priorities"
                untouched = np.ones(cap, bool); untouched[slots[g]] = False
                assert np.array_equal(pr1[g, untouched], pr0[g, untouched])
                assert pmax1[g] == max(pmax0[g], pr1[g, slots[g]].max())
        if tie.any():
            load()
            continue
        close(metrics[:, 0], out["loss"], what=f"step {step} loss")
        g64 = branch_gradients([p.numpy() for p in th0], S, A_, out["y"], loss, dbg["dh1"] != 0, dbg["dh2"] != 0,
                               weights=isw)
        alpha_t, eps_t = adam_scalars(t, 5e-4, "keras")
        for i in range(n):
            got, gm, gv = grp.get_weights(i, "online"), grp.get_weights(i, "m"), grp.get_weights(i, "v")
            for k in range(6):
                gk = torch.as_tensor(g64[k][i])
                adam_close(got[k].numpy(), th0[k][i], m0[k][i], v0[k][i], gk, alpha_t, eps_t, what=f"step {step} net {i} theta[{k}]")
                close(gm[k].numpy(), (m0[k][i] + (gk - m0[k][i]) * np.float32(0.1)).numpy(), what=f"step {step} net {i} m[{k}]")
                close(gv[k].numpy(), (v0[k][i] + (gk * gk - v0[k][i]) * np.float32(0.001)).numpy(), rtol=2 * RTOL,
                      what=f"step {step} net {i} v[{k}]")
        load()                                          # keep the trajectories together: later steps test the kernel


def chained_step_equals_stage_by_stage_step(config):
    from dmdqn_b200 import _native as N
    n, cap, b = 40, 160, 128
    kw = dict(h=256, precision="tf32x3", seed=2, **config)
    a, c = replay_group(n, cap, b, **kw), replay_group(n, cap, b, **kw)
    for g in (a, c):
        fill_rings(g, cap + 3, seed=8)
    rng = np.random.default_rng(9)
    for it in range(4):
        w = draw_words(rng, n, b)
        ma = a.learn(w).clone()
        for stage in (1, 2, 4, 8):
            N.check(c.lib.dmdqn_learn_stages(C.byref(c.dims), C.byref(c.hp), C.byref(c.replay), C.byref(c.nets), w.data_ptr(),
                                             None, c.metrics.data_ptr(), c.workspace.data_ptr(), c.workspace.numel(), stage,
                                             torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert torch.equal(ma, c.metrics), f"step {it}: metrics differ"
        for name in state_names(a):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name} differs"


def captured_learn_equals_plain_learn(config):
    """With prioritized replay beta anneals over the captured steps (0.6, 0.8, 1.0, 1.0, ...): the graph reads it on the
    device."""
    n, cap, b = 16, 300, 64
    kw = dict(h=256, precision="tf32x3", seed=9, **config)
    if kw.get("sample_mode") == "prioritized":
        kw["per_beta_steps"] = 3
    a, c = replay_group(n, cap, b, **kw), replay_group(n, cap, b, **kw)
    for g in (a, c):
        fill_rings(g, cap, seed=10)
    replay, draws = c.capture_learn()
    a.learn(draws.clone())                             # the capture's warm-up step, on a
    rng = np.random.default_rng(11)
    for it in range(5):
        w = draw_words(rng, n, b)
        draws.copy_(w)
        mc = replay().clone()
        ma = a.learn(w).clone()
        torch.cuda.synchronize()
        assert torch.equal(ma, mc), f"step {it}: metrics differ"
        if a.prioritized:
            assert torch.equal(a.debug_views()["is_weights"], c.debug_views()["is_weights"])
        for name in state_names(a, "learn_step"):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name} differs"


def captured_step_host_equals_step_host(config):
    n, cap, b = 12, 200, 64
    kw = dict(h=256, precision="tf32x3", seed=5, **config)
    a, c = replay_group(n, cap, b, **kw), replay_group(n, cap, b, **kw)
    for g in (a, c):
        fill_rings(g, cap - 10, seed=12)
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
        assert torch.equal(ma, mc), f"step {it}: metrics differ"
        for name in state_names(a, "obs", "done_ring"):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name} differs"


def one_group_of_eight_equals_two_groups_of_four(config):
    n, cap, b = 8, 300, 128
    big = replay_group(n, cap, b, h=256, precision="tf32x3", seed=14, **config)
    fill_rings(big, [cap + 5, cap, 250, 400, 300, 129, 1000, 301], seed=15)
    halves = [replay_group(4, cap, b, h=256, precision="tf32x3", seed=99, **config) for _ in range(2)]
    for k, hg in enumerate(halves):
        copy_state(hg, big, slice(4 * k, 4 * k + 4))
    rng = np.random.default_rng(16)
    for it in range(4):
        w = draw_words(rng, n, b)
        mb = big.learn(w).clone()
        mh = torch.cat([hg.learn(w[4 * k:4 * k + 4].contiguous()).clone() for k, hg in enumerate(halves)])
        torch.cuda.synchronize()
        assert torch.equal(mb, mh), f"step {it}: metrics differ"
        for name in state_names(big):
            assert torch.equal(getattr(big, name), torch.cat([getattr(hg, name) for hg in halves])), f"step {it}: {name}"


def train_loop_learns_from_the_config_alone(config, mode):
    """train_agents needs nothing but the config: both call patterns learn with prioritized replay (the learn steps move
    the priorities of the slots they drew) or with n-step returns."""
    from dmdqn_b200.train import PRESETS, train_agents
    cfg = dict(PRESETS["shipped_train_py"])
    cfg.update(max_sim_time=600.0, backend="fake", grid_rows=3, grid_cols=3, fake_traci_seed=11, batch_size=16,
               nn_layers=[64, 64], precision="auto", **config)
    if config.get("sample_mode") == "prioritized":
        cfg["per_beta_steps"] = 10
    history, agents, group = train_agents(cfg, episodes=1, mode=mode, seed=3, learn=True)
    t = len(history)
    assert t > 16 and np.all(group.learn_step.cpu().numpy() == t - 15)      # one learn step per step once 16 are stored
    assert any(h["total_loss"] != 0 for h in history)
    assert int(group.debug_views()["tc_error"][0]) == 0
    if config.get("sample_mode") == "prioritized":
        assert group.prioritized and group.priority.shape == (9, group.capacity)
        pr = group.priority.cpu().numpy()
        assert np.all(pr[:, :t] > 0) and np.all(pr[:, t:] == 0)
        assert np.any(pr[:, :t] != 1.0)                                        # priorities from TD errors, not only the push rule
    else:
        assert group.hp.n_step == 3
        assert np.all(np.isfinite([h["total_loss"] for h in history]))
        if mode == "batched":                          # the last step's targets bootstrap up to three steps ahead
            dbg = group.debug_views()
            g = 0.99
            assert np.any(dbg["discount"].cpu().numpy() == np.float32(g * g * g))
            assert torch.any(dbg["next_rows"] != dbg["rows"])
