"""Global-norm gradient clipping on the GPU (config ``global_clipnorm``: dmdqn_learn_grads -> dmdqn_clip_adam_apply):
the gradient block against the float64 branch gradients, the norm against numpy's float64 norm of the device's own block,
the scale and the clipped Adam step bit for bit against dmdqn_adam_apply on the scaled block, the unclipped step, inactive
and poisoned-free networks, prioritized replay with n-step targets, shared parameters and the execution orders.  Run on
the B200 box: pytest -m gpu"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.dqn import adam_scalars
from parity_util import (PER, RTOL, adam_close, branch_gradients, captured_learn_equals_plain_learn, captured_step_host_equals_step_host,
                         close, draw_words, fill_rings, one_group_of_eight_equals_two_groups_of_four, replay_group,
                         train_loop_learns_from_the_config_alone, ulps)

pytestmark = pytest.mark.gpu
STATE = ("theta", "theta_tgt", "adam_m", "adam_v")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _save(grp):
    names = STATE + ("learn_step",) + (("priority", "priority_max") if grp.prioritized else ())
    return {k: getattr(grp, k).clone() for k in names}, grp.learn_step_host.copy()


def _restore(grp, saved, names=None):
    state, host = saved
    for k in names or state:
        getattr(grp, k).copy_(state[k])
    grp.learn_step_host[:] = host


def _adam_apply(grp, grads):
    from dmdqn_b200 import _native as N
    N.check(grp.lib.dmdqn_adam_apply(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), grads.data_ptr(),
                                     grp.workspace.data_ptr(), grp.workspace.numel(), _stream()))


def _learn_grads(grp, words, grads, mask=None):
    from dmdqn_b200 import _native as N
    N.check(grp.lib.dmdqn_learn_grads(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.replay), C.byref(grp.nets),
                                      words.data_ptr(), None if mask is None else mask.data_ptr(), grp.batch_size,
                                      grads.data_ptr(), grp.metrics.data_ptr(), grp.workspace.data_ptr(), grp.workspace.numel(),
                                      _stream()))


def _block_norms(grp, grads):
    p = int(grp.layout.b3) + 4
    g = grads[:, :p].cpu().numpy().astype(np.float64)
    return np.sqrt((g * g).sum(axis=1))


def _check_scaled_update(grp, before, after, grads, norms64, c, what):
    """The clipped step equals dmdqn_adam_apply on grads * s' with s' within 1 ulp of (float)(c / max(n, c)) (numpy's
    float64 norm of the device's block): theta, m, v and the target, bit for bit.  s' = 1 exactly for an unclipped network."""
    s_ref = np.array([np.float32(c / max(n, c)) for n in norms64], np.float32)
    cands = [s_ref] if np.all(s_ref == 1) else [s_ref, np.nextafter(s_ref, np.float32(0)), np.nextafter(s_ref, np.float32(2))]
    matched = np.zeros(grp.n_nets, bool)
    for s in cands:
        _restore(grp, before, STATE)
        scaled = grads * torch.as_tensor(s, device=grads.device)[:, None]
        _adam_apply(grp, scaled)
        torch.cuda.synchronize()
        for i in range(grp.n_nets):
            if all(torch.equal(getattr(grp, k)[i], after[0][k][i]) for k in STATE):
                matched[i] = True
    assert matched.all(), f"{what}: networks {np.nonzero(~matched)[0]} match no scale within 1 ulp"
    unclipped = s_ref == 1
    if unclipped.any():                                   # those match dmdqn_adam_apply on the raw block itself
        _restore(grp, before, STATE)
        _adam_apply(grp, grads)
        for i in np.nonzero(unclipped)[0]:
            for k in STATE:
                assert torch.equal(getattr(grp, k)[i], after[0][k][i]), f"{what}: unclipped net {i} {k}"
    _restore(grp, after)
    return s_ref


# ------------------------------------------------------------------ 1. parity -------------------------------------------
@pytest.mark.parametrize("h,precision,loss,double_dqn,tau,mode,n_step", [
    (64, "fp32", "mse", True, None, "fisher_yates", 1), (64, "fp32", "huber", False, 0.01, "fisher_yates", 1),
    (256, "fp32", "huber", True, None, "fisher_yates", 1), (256, "fp32", "mse", False, 0.01, "fisher_yates", 1),
    (256, "tf32x3", "mse", True, None, "fisher_yates", 1), (256, "tf32x3", "huber", False, 0.01, "fisher_yates", 1),
    (64, "fp32", "mse", True, None, "prioritized", 3), (256, "tf32x3", "huber", True, None, "prioritized", 3)])
def test_clipped_step_matches_the_oracle_gradient_and_the_scaled_adam_step(h, precision, loss, double_dqn, tau, mode, n_step):
    n, cap, b = 3, 200, 128
    grp = replay_group(n, cap, b, h=h, precision=precision, loss=loss, double_dqn=double_dqn, tau=tau, sample_mode=mode,
                       n_step=n_step, global_clipnorm=1.0)
    fill_rings(grp, [cap + 40, 150, cap], seed=h + 1, done_rate=0.1)
    twin = replay_group(n, cap, b, h=h, precision=precision, loss=loss, double_dqn=double_dqn, tau=tau, sample_mode=mode,
                        n_step=n_step)                   # the same steps without clipping: K4a is unchanged
    fill_rings(twin, [cap + 40, 150, cap], seed=h + 1, done_rate=0.1)
    rng = np.random.default_rng(h + n_step)
    obs, act = grp.obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    clipped_seen = unclipped_seen = 0
    for step in range(6):                                # target_update_frequency 3: steps 3 and 6 copy the target
        words = draw_words(rng, n, b)
        before = _save(grp)
        grp.global_clipnorm = 1e30                       # a probe of this step's norms
        grp.learn(words)
        probe = grp.grad_norms.cpu().numpy()
        _restore(grp, before)
        c = float(max(np.median(probe) / 4, probe.min() * 1.001))
        grp.global_clipnorm = c
        th0 = [grp.get_weights(i, "online") for i in range(n)]
        m0, v0 = [grp.get_weights(i, "m") for i in range(n)], [grp.get_weights(i, "v") for i in range(n)]
        pr0 = None if grp.priority is None else grp.priority.clone()
        grp.grads.fill_(float("nan"))                    # every element of the block must be written
        metrics = grp.learn(words).clone()
        twin.learn(words)
        torch.cuda.synchronize()
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        assert int(dbg["tc_error"][0]) == 0
        grads = grp.grads.clone()
        norms = grp.grad_norms.cpu().numpy()
        assert np.all(np.isfinite(grads.cpu().numpy()[:, :int(grp.layout.b3) + 4])), f"step {step}: unwritten gradient"
        n64 = _block_norms(grp, grads)
        assert ulps(norms, n64.astype(np.float32)).max() <= 1, f"step {step}: norms {norms} vs {n64}"
        assert torch.equal(metrics, twin.metrics), f"step {step}: metrics"
        if pr0 is not None:                              # priorities come from K4a: bit-identical to the unclipped step
            assert torch.equal(grp.priority, twin.priority) and torch.equal(grp.priority_max, twin.priority_max)
        after = _save(grp)
        s = _check_scaled_update(grp, before, after, grads, n64, c, f"step {step}")
        clipped_seen += int((s < 1).sum()); unclipped_seen += int((s == 1).sum())
        # the gradient block against the exact gradients on the kernel's own branch
        slots = dbg["rows"] % cap
        S = np.stack([obs[g, slots[g]] for g in range(n)])
        A_ = np.stack([act[g, slots[g]] for g in range(n)])
        isw = dbg["is_weights"] if mode == "prioritized" else None
        g64 = branch_gradients([np.stack([th0[i][k].numpy() for i in range(n)]) for k in range(6)], S, A_, dbg["y"], loss,
                               dbg["dh1"] != 0, dbg["dh2"] != 0, weights=isw)
        alpha_t, eps_t = adam_scalars(int(grp.learn_step_host[0]), 5e-4, "keras")
        for i in range(n):
            got = grp.unpack(grads[i])
            th1, m1, v1 = grp.get_weights(i, "online"), grp.get_weights(i, "m"), grp.get_weights(i, "v")
            for k in range(6):
                w = f"step {step} net {i}"
                close(got[k].numpy(), g64[k][i], rtol=10 * RTOL, what=f"{w} grad[{k}]")
                # the existing 1e-5 bars of the learn step, on the scaled gradient
                gk = torch.as_tensor(g64[k][i]) * s[i]
                adam_close(th1[k].numpy(), th0[i][k], m0[i][k], v0[i][k], gk, alpha_t, eps_t, what=f"{w} theta[{k}]")
                close(m1[k].numpy(), (m0[i][k] + (gk - m0[i][k]) * np.float32(0.1)).numpy(), what=f"{w} m[{k}]")
                close(v1[k].numpy(), (v0[i][k] + (gk * gk - v0[i][k]) * np.float32(0.001)).numpy(), rtol=2 * RTOL,
                      what=f"{w} v[{k}]")
        for k in STATE:                                  # keep the twin on the clipped trajectory
            getattr(twin, k).copy_(getattr(grp, k))
    assert clipped_seen > 0 and unclipped_seen > 0


# ------------------------------------------------------------------ 2. threshold above every norm -----------------------
@pytest.mark.parametrize("h,precision", [(64, "fp32"), (256, "fp32"), (256, "tf32x3")])
def test_a_threshold_above_every_norm_is_learn_grads_then_adam_apply_bit_for_bit(h, precision):
    n, cap, b = 4, 200, 128
    kw = dict(h=h, precision=precision, loss="huber", seed=3)
    clip, parts, fused = (replay_group(n, cap, b, global_clipnorm=1e30, **kw), replay_group(n, cap, b, **kw),
                          replay_group(n, cap, b, **kw))
    for g in (clip, parts, fused):
        fill_rings(g, [cap, cap + 7, 180, cap], seed=4)
    grads = torch.zeros_like(parts.theta)
    rng = np.random.default_rng(5)
    identical_to_fused = True
    for step in range(4):
        w = draw_words(rng, n, b)
        mc = clip.learn(w).clone()
        _learn_grads(parts, w, grads)
        _adam_apply(parts, grads)
        mf = fused.learn(w).clone()
        torch.cuda.synchronize()
        assert torch.equal(mc, parts.metrics), f"step {step}: metrics"
        for k in STATE + ("learn_step",):
            assert torch.equal(getattr(clip, k), getattr(parts, k)), f"step {step}: {k}"
        assert torch.equal(clip.grad_norms.cpu(), torch.as_tensor(_block_norms(clip, grads).astype(np.float32))) or \
            ulps(clip.grad_norms.cpu().numpy(), _block_norms(clip, grads).astype(np.float32)).max() <= 1
        close(mc.cpu().numpy(), mf.cpu().numpy(), what=f"step {step}: metrics against dmdqn_learn")
        for k in STATE:
            close(getattr(clip, k).cpu().numpy(), getattr(fused, k).cpu().numpy(), what=f"step {step}: {k} against dmdqn_learn")
            identical_to_fused &= torch.equal(getattr(clip, k), getattr(fused, k))
            getattr(fused, k).copy_(getattr(clip, k))    # the 1e-5 bar per step, not over a drifting trajectory
    print(f"[{h} {precision}] clipped step with no clipping bit-identical to dmdqn_learn: {identical_to_fused}")
    if precision == "fp32":                              # the FFMA K4b applies adam_elem to the same sums
        assert identical_to_fused


# ------------------------------------------------------------------ 4. inactive networks --------------------------------
@pytest.mark.parametrize("h,precision", [(64, "fp32"), (256, "tf32x3")])
def test_inactive_networks_are_untouched_and_report_norm_zero(h, precision):
    n, cap, b = 4, 200, 128
    grp = replay_group(n, cap, b, h=h, precision=precision, global_clipnorm=1e-3)
    fill_rings(grp, [cap, 60, cap, cap], seed=6)          # network 1: ring not full yet
    mask = torch.tensor([1, 1, 0, 1], dtype=torch.uint8)  # network 2: masked out
    before = {k: getattr(grp, k).clone() for k in STATE}
    grp.grad_norms.fill_(float("nan"))
    m = grp.learn(draw_words(np.random.default_rng(7), n, b), mask=mask).cpu().numpy()
    norms = grp.grad_norms.cpu().numpy()
    assert np.all(norms[[1, 2]] == 0) and np.all(norms[[0, 3]] > 1e-3)
    assert np.all(m[[1, 2]] == 0) and np.all(m[[0, 3], 7] == 1)
    for k in STATE:
        for i in (1, 2):
            assert torch.equal(getattr(grp, k)[i], before[k][i]), f"net {i}: {k} changed"
        for i in (0, 3):
            assert not torch.equal(grp.theta[i], before["theta"][i])


# ------------------------------------------------------------------ 6. shared parameters --------------------------------
def _shared(h, n_agents, batch, cap, seed, precision="fp32", clip=0.05):
    grp = replay_group(n_agents, cap, batch, h=h, precision=precision, share_parameters=True, global_clipnorm=clip,
                       target_update_frequency=2, seed=1)
    fill_rings(grp, cap + 2, seed=seed)
    return grp


def test_shared_parameters_world_one_matches_the_big_batch_clipped_oracle():
    import clip_oracle as O
    from dmdqn_b200.parallel import SharedParameterStep
    from oracle import replay as R
    h, n_agents, b, cap, clip = 64, 8, 256, 40, 0.05
    grp = _shared(h, n_agents, b, cap, seed=30, clip=clip)
    stk = O.ClipStackedOracle(1, 89, [h, h], 4, gamma=0.99, learning_rate=5e-4, target_update_frequency=2, seed0=9)
    for which, src in (("online", stk.online), ("target", stk.target)):
        grp.set_weights(0, [p[0] for p in src], which)
    step = SharedParameterStep.for_group(grp)
    assert step.fused_apply is None                       # clipping takes the NCCL path
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    rng = np.random.default_rng(31)
    for it in range(3):
        words = rng.integers(0, 2**32, (1, b), dtype=np.uint64).astype(np.uint32)
        grp.draw_words = lambda shape, w=words: torch.as_tensor(w.view(np.int32)).to(grp.device)
        step.step()
        torch.cuda.synchronize()
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        rows = dbg["rows"][0]
        ag, sl = rows // cap, rows % cap
        done = (dbg["discount"][0] == 0).astype(np.float32)
        out = stk.learn_on_batch(obs[ag, sl][None], act[ag, sl][None], dbg["r_hat"], nobs[ag, sl][None], done[None],
                                 discounts=dbg["discount"], global_clipnorm=clip)
        assert out["norms"][0] > clip
        assert abs(float(grp.grad_norms[0]) - out["norms"][0]) <= 1e-5 * out["norms"][0]
        for k, (got, ref) in enumerate(zip(grp.get_weights(0, "online"), stk.online)):
            close(got.numpy(), ref[0].numpy(), what=f"step {it} theta[{k}]")
        for k, (got, ref) in enumerate(zip(grp.get_weights(0, "target"), stk.target)):
            close(got.numpy(), ref[0].numpy(), what=f"step {it} target[{k}]")
        for which, src in (("online", stk.online), ("target", stk.target), ("m", stk.adam_m), ("v", stk.adam_v)):
            grp.set_weights(0, [p[0] for p in src], which)


@pytest.mark.parametrize("world", [2, 3])
def test_simulated_ranks_stay_bit_identical_after_the_clipped_step(world):
    from dmdqn_b200.parallel import SharedParameterStep
    h, n_agents, b, cap = 256, 2, 128, 150
    ranks = [_shared(h, n_agents, b, cap, seed=40 + 17 * r, precision="tf32x3") for r in range(world)]
    steps = [SharedParameterStep.for_group(g) for g in ranks]
    streams = [torch.cuda.Stream() for _ in range(world)]
    rng = np.random.default_rng(41)
    for it in range(3):
        torch.cuda.synchronize()
        blocks = []
        for r in range(world):
            words = rng.integers(0, 2**32, (1, b), dtype=np.uint64).astype(np.uint32)
            ranks[r].draw_words = lambda shape, w=words: torch.as_tensor(w.view(np.int32)).cuda()
            with torch.cuda.stream(streams[r]):
                blocks.append(steps[r].local_grads(b * world)[0].clone())
        torch.cuda.synchronize()
        total = blocks[0].clone()
        for blk in blocks[1:]:                            # rank order, as the all-reduce sums
            total += blk
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                steps[r].apply(total)
        torch.cuda.synchronize()
        for g in ranks:
            g.check_errors()
        norms = [float(g.grad_norms[0]) for g in ranks]
        assert norms[0] > 0.05 and len(set(norms)) == 1, norms
        for r in range(1, world):
            for k in STATE:
                assert torch.equal(getattr(ranks[r], k), getattr(ranks[0], k)), f"step {it}: replica {r} {k} diverged"


# ------------------------------------------------------------------ 7. execution orders ---------------------------------
CLIP = {"global_clipnorm": 0.05}


def test_captured_learn_equals_plain_learn():
    captured_learn_equals_plain_learn(CLIP)


def test_captured_step_host_equals_step_host():
    captured_step_host_equals_step_host(CLIP)


def test_one_group_of_eight_equals_two_groups_of_four():
    one_group_of_eight_equals_two_groups_of_four(CLIP)
    one_group_of_eight_equals_two_groups_of_four({**CLIP, **PER, "n_step": 3})


def test_two_runs_give_the_same_bits():
    runs = []
    for _ in range(2):
        grp = replay_group(8, 300, 128, h=256, precision="tf32x3", seed=14, **CLIP)
        fill_rings(grp, 300, seed=15)
        rng = np.random.default_rng(16)
        for _ in range(3):
            grp.learn(draw_words(rng, 8, 128))
        torch.cuda.synchronize()
        runs.append([getattr(grp, k).clone() for k in STATE + ("grad_norms", "metrics")])
    for a, c in zip(*runs):
        assert torch.equal(a, c)


# ------------------------------------------------------------------ 8. the training loop -----------------------------------
@pytest.mark.parametrize("mode", ["batched", "per_agent"])
def test_train_loop_clips_from_the_config_alone(mode):
    train_loop_learns_from_the_config_alone({"global_clipnorm": 10.0, "n_step": 3}, mode)
