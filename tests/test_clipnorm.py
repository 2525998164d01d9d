"""CPU checks of global-norm gradient clipping (config ``global_clipnorm``, dmdqn_clip_adam_apply): the restated clip
against torch's ``clip_grad_norm_``, the oracle's clipped learn step against autograd, the config key, the refusals that
need no GPU, and the shared-parameter step with clipping over gloo with the oracle standing in for the kernels."""
import ctypes as C
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import clip_oracle as O
from replay_oracle import ReplayStackedOracle
from dmdqn_b200.parallel import SharedParameterStep


def _blocks(rng, scale):
    shapes = [(89, 32), (32,), (32, 32), (32,), (32, 4), (4,)]
    return [(rng.standard_normal(s) * scale).astype(np.float32) for s in shapes]


@pytest.mark.parametrize("scale,c", [(1.0, 0.5), (1.0, 3.0), (0.01, 1.0), (100.0, 10.0), (0.05, 0.5)])
def test_clip_matches_torch_clip_grad_norm(scale, c):
    rng = np.random.default_rng(int(scale * 1000) + int(c * 7))
    for _ in range(4):
        g = _blocks(rng, scale)
        n, s = O.clip_scale(g, c)
        ref = math.sqrt(sum(float((x.astype(np.float64) ** 2).sum()) for x in g))
        assert n == pytest.approx(ref, rel=1e-15)
        params = [torch.zeros(x.shape, requires_grad=True) for x in g]
        for p, x in zip(params, g):
            p.grad = torch.as_tensor(x.copy())
        total = torch.nn.utils.clip_grad_norm_(params, c)
        assert float(total) == pytest.approx(n, rel=1e-6)
        for p, x in zip(params, g):
            ours = x * s
            if n <= c:                                  # no clipping: s is exactly 1 and the gradient is untouched
                assert s == np.float32(1.0) and np.array_equal(ours, x)
            else:                                       # torch scales by c / (n + 1e-6); n > 1 in these cases
                np.testing.assert_allclose(ours, p.grad.numpy(), rtol=2e-6, atol=0)


def test_clip_of_a_non_finite_gradient_applies_no_scaling():
    g = [np.array([1.0, np.inf], np.float32)]
    n, s = O.clip_scale(g, 1.0)
    assert not np.isfinite(n) and s == np.float32(1.0)
    n, s = O.clip_scale([np.array([np.nan], np.float32)], 1.0)
    assert np.isnan(n) and s == np.float32(1.0)


@pytest.mark.parametrize("loss", ["mse", "huber"])
def test_oracle_clipped_step_is_autograd_then_clip_grad_norm_then_adam(loss):
    from oracle.dqn import StackedOracle, adam_scalars, adam_update_, loss_and_grad
    rng = np.random.default_rng(5)
    n, b, h = 3, 32, 32
    s, s2 = rng.integers(-1, 20, (n, b, 89)).astype(np.float32), rng.integers(-1, 20, (n, b, 89)).astype(np.float32)
    a, r = rng.integers(0, 4, (n, b)), (rng.standard_normal((n, b)) * 30).astype(np.float32)
    d = (rng.random((n, b)) < 0.2).astype(np.float32)
    kw = dict(gamma=0.99, learning_rate=5e-4, loss=loss, target_update_frequency=3, seed0=21)
    stk, ref = O.ClipStackedOracle(n, 89, [h, h], 4, **kw), StackedOracle(n, 89, [h, h], 4, **kw)
    for step in range(3):
        y, _, _ = ref.td_targets(r, s2, d)
        params = [p.detach().requires_grad_(True) for p in ref.online]
        q = ref.forward(params, torch.as_tensor(s))
        pred = torch.gather(q, 2, torch.as_tensor(a)[..., None])[..., 0]
        terms, _ = loss_and_grad(pred, y, loss)
        grads = torch.autograd.grad(terms.mean(dim=1).sum(), params)
        norms = [float(torch.sqrt(sum((g[i].double() ** 2).sum() for g in grads))) for i in range(n)]
        c = float(np.median(norms)) * (0.5 if step else 2.0)       # at least one network clips, at step 0 not all
        with torch.no_grad():
            for i in range(n):
                gi = [torch.zeros(g[i].shape, requires_grad=True) for g in grads]
                for p, g in zip(gi, grads):
                    p.grad = g[i].clone()
                torch.nn.utils.clip_grad_norm_(gi, c)
                ref.learn_step[i] += 1
                alpha, eps = adam_scalars(int(ref.learn_step[i]), ref.lr)
                for p, g, m, v in zip(ref.online, gi, ref.adam_m, ref.adam_v):
                    adam_update_(p[i], g.grad, m[i], v[i], alpha, eps)
                if ref.learn_step[i] % ref.freq == 0:
                    for t, o in zip(ref.target, ref.online):
                        t[i].copy_(o[i])
        out = stk.learn_on_batch(s, a, r, s2, d, global_clipnorm=c)
        np.testing.assert_allclose(out["norms"], norms, rtol=1e-6)        # the weights differ by torch's 1e-6
        for x, yv in zip(stk.online + stk.target, ref.online + ref.target):
            np.testing.assert_allclose(x.numpy(), yv.numpy(), rtol=1e-6, atol=1e-6 * float(yv.abs().max()))


def test_oracle_without_a_clipnorm_or_with_one_above_every_norm_is_the_plain_step_bit_for_bit():
    rng = np.random.default_rng(8)
    n, b = 2, 16
    s, s2 = rng.integers(-1, 20, (n, b, 89)).astype(np.float32), rng.integers(-1, 20, (n, b, 89)).astype(np.float32)
    a, r = rng.integers(0, 4, (n, b)), rng.standard_normal((n, b)).astype(np.float32)
    d = (rng.random((n, b)) < 0.2).astype(np.float32)
    kw = dict(gamma=0.99, learning_rate=5e-4, loss="mse", target_update_frequency=3, seed0=2)
    plain = ReplayStackedOracle(n, 89, [32, 32], 4, **kw)
    none, high = (O.ClipStackedOracle(n, 89, [32, 32], 4, **kw) for _ in range(2))
    for _ in range(3):
        plain.learn_on_batch(s, a, r, s2, d)
        none.learn_on_batch(s, a, r, s2, d, global_clipnorm=None)
        out = high.learn_on_batch(s, a, r, s2, d, global_clipnorm=1e30)
        assert np.all(out["norms"] > 0)
    for o in (none, high):
        for mine, ref in zip(o.online + o.target + o.adam_m + o.adam_v, plain.online + plain.target + plain.adam_m + plain.adam_v):
            assert torch.equal(mine, ref)
        assert np.array_equal(o.learn_step, plain.learn_step)


def test_config_default_and_yaml_key():
    from dmdqn_b200 import train
    from dmdqn_b200.group import DEFAULTS
    assert DEFAULTS["global_clipnorm"] is None
    assert train.load_config()["global_clipnorm"] is None


@pytest.mark.parametrize("value", [0, 0.0, -1, -1e-3, float("nan"), float("inf"), float("-inf"), "10", True, [1.0]])
def test_agent_group_refuses_a_clipnorm_that_is_not_a_positive_finite_number(value):
    from dmdqn_b200.group import AgentGroup
    with pytest.raises(ValueError, match="global_clipnorm"):
        AgentGroup(4, {"nn_layers": [64, 64], "global_clipnorm": value})


@pytest.fixture(scope="module")
def lib():
    from dmdqn_b200 import _native as N
    from dmdqn_b200 import build as B
    B.build()
    return N.lib()


def test_native_clip_adam_apply_refuses_bad_arguments_before_launching_anything(lib):
    from dmdqn_b200 import _native as N
    dims = N.Dims(4, 4, 89, 96, 64, 4, 32, 100)
    nbytes = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(dims), C.byref(nbytes)))
    ws = (C.c_uint8 * 256)()           # never touched: validation fails before anything is launched
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 1000, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100)
    nets = N.Nets(1, 1, 1, 1, 1)
    call = lambda c, nets=nets, grads=C.addressof(ws): lib.dmdqn_clip_adam_apply(
        C.byref(dims), C.byref(hp), C.byref(nets), grads, c, None, C.addressof(ws), nbytes.value, None)
    for c in (0.0, -1.0, float("nan"), float("inf"), float("-inf")):
        assert call(c) == N.ERR_ARG, c
        assert "global_clipnorm" in lib.dmdqn_last_error().decode(), c
    assert call(1.0, grads=None) == N.ERR_ARG and "NULL" in lib.dmdqn_last_error().decode()
    assert call(1.0, nets=N.Nets(1, 1, None, 1, 1)) == N.ERR_ARG and "NULL" in lib.dmdqn_last_error().decode()
    assert lib.dmdqn_clip_adam_apply(C.byref(dims), None, C.byref(nets), C.addressof(ws), 1.0, None, C.addressof(ws),
                                     nbytes.value, None) == N.ERR_ARG
    assert lib.dmdqn_clip_adam_apply(C.byref(dims), C.byref(hp), C.byref(nets), C.addressof(ws), 1.0, None, C.addressof(ws),
                                     nbytes.value - 1, None) == N.ERR_WORKSPACE


def test_fused_shared_step_with_clipping_is_refused():
    class Shared:                       # what for_group reads before it touches a device
        shared, global_clipnorm = True, 1.0
    with pytest.raises(ValueError, match="does not clip"):
        SharedParameterStep.for_group(Shared(), fused=True)


# ------------------------------------------------------------------ gloo, world size 2 ----------------------------------
H, B_GLOBAL, CLIP = 64, 64, 0.05


def _data():
    rng = np.random.default_rng(0)
    S = rng.integers(-1, 20, (1, B_GLOBAL, 89)).astype(np.float32)
    S2 = rng.integers(-1, 20, (1, B_GLOBAL, 89)).astype(np.float32)
    A_ = rng.integers(0, 4, (1, B_GLOBAL)); R = (rng.standard_normal((1, B_GLOBAL)) * 20).astype(np.float32)
    D = (rng.random((1, B_GLOBAL)) < 0.1).astype(np.float32)
    return S, A_, R, S2, D


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from oracle.dqn import StackedOracle, adam_scalars, adam_update_, loss_and_grad
        torch.set_num_threads(1)
        b_local = B_GLOBAL // world
        S, A_, R, S2, D = _data()
        sl = slice(rank * b_local, (rank + 1) * b_local)
        stk = StackedOracle(1, 89, [H, H], 4, seed0=3)
        norms = []

        def local_grads(global_batch):
            y, _, _ = stk.td_targets(R[:, sl], S2[:, sl], D[:, sl])
            params = [p.detach().requires_grad_(True) for p in stk.online]
            qv = stk.forward(params, torch.as_tensor(S[:, sl]))
            pred = torch.gather(qv, 2, torch.as_tensor(A_[:, sl])[..., None])[..., 0]
            terms, _ = loss_and_grad(pred, y, "mse")
            loss = terms.sum(dim=1) / global_batch
            grads = torch.autograd.grad(loss.sum(), params)
            metrics = torch.zeros(1, 8); metrics[0, 0] = loss.detach()[0]
            return torch.cat([g.reshape(-1) for g in grads]), metrics

        def apply(flat):                # dmdqn_clip_adam_apply on the all-reduced block
            n, s = O.clip_scale([flat.numpy()], CLIP)
            norms.append(n)
            flat = flat * s if s != 1 else flat
            stk.learn_step[0] += 1
            alpha, eps = adam_scalars(int(stk.learn_step[0]), stk.lr)
            off = 0
            with torch.no_grad():
                for p, m, v in zip(stk.online, stk.adam_m, stk.adam_v):
                    k = p.numel()
                    adam_update_(p, flat[off:off + k].view_as(p), m, v, alpha, eps)
                    off += k

        step = SharedParameterStep(local_grads, apply, b_local)
        for _ in range(2):
            step.step()
        q.put((rank, norms, [p.clone().numpy() for p in stk.online]))
    finally:
        dist.destroy_process_group()


def test_shared_parameter_clipped_step_equals_single_process_big_batch_clipped_step():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    S, A_, R, S2, D = _data()
    ref = O.ClipStackedOracle(1, 89, [H, H], 4, seed0=3)
    ref_norms = [ref.learn_on_batch(S, A_, R, S2, D, global_clipnorm=CLIP)["norms"][0] for _ in range(2)]
    assert min(ref_norms) > CLIP                        # both steps clip
    for rank, norms, weights in results:
        np.testing.assert_allclose(norms, ref_norms, rtol=1e-5)
        for w, r in zip(weights, ref.online):
            np.testing.assert_allclose(w, r.numpy(), rtol=1e-5, atol=1e-6)
    assert results[0][1] == results[1][1]               # the same norm on every rank ...
    for w0, w1 in zip(results[0][2], results[1][2]):    # ... so the replicas stay identical
        assert np.array_equal(w0, w1)
