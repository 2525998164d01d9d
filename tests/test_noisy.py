"""Noisy networks on the CPU (config ``noisy``): the Philox restatement against Random123's known-answer vectors, the noisy
oracle against a torch.nn factorized NoisyLinear module, the fold and gradient identities, the zero padding factors, the
sigma init and the noise keys, the config keys and refusals, and the shared-parameter noisy step over gloo with the oracle
standing in for the kernels."""
import ctypes as C
import math
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import noisy_oracle as O
from dmdqn_b200.parallel import SharedParameterStep


@pytest.mark.parametrize("key,ctr,want", [
    ((0, 0), (0, 0, 0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff, 0xffffffff), (0xffffffff,) * 4, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0xa4093822, 0x299f31d0), (0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_restatement_reproduces_random123_known_answers(key, ctr, want):
    assert tuple(int(x) for x in O.philox4x32_10(ctr, key)) == want


def test_factors_are_standard_normal_through_f_and_keyed_by_every_counter_field():
    z = O.box_muller(*O.philox4x32_10((np.arange(200000), 0, 0, O.NOIS), (1, 2))[:2])
    assert abs(float(z.mean())) < 0.01 and abs(float(z.std()) - 1) < 0.01
    f = O.factor(z)
    assert np.array_equal(np.sign(f), np.sign(z)) and np.allclose(f * f, np.abs(z), rtol=1e-6)
    base = O.factor_vector(7, 3, 0, 5, 64, 64)
    for other in (O.factor_vector(8, 3, 0, 5, 64, 64), O.factor_vector(7, 2, 0, 5, 64, 64),
                  O.factor_vector(7, 3, 1, 5, 64, 64), O.factor_vector(7, 3, 0, 6, 64, 64)):
        assert not np.any(base == other)


def _rec(dp, h):
    off = np.cumsum([0, dp, h, h, h, h, 4, h, 4])
    return SimpleNamespace(**dict(zip(("w1_in", "w1_out", "w2_in", "w2_out", "w3_in", "w3_out", "v_in", "v_out"), off[:8])),
                           stride=int((off[8] + 31) // 32 * 32))


@pytest.mark.parametrize("obs_dim,dp,a", [(89, 96, 4), (89, 96, 3), (30, 32, 2)])
def test_padding_factors_are_exactly_zero(obs_dim, dp, a):
    rec = _rec(dp, 64)
    r = O.noise_record(0x1234_5678_9abc_def0, 3, 1, rec, obs_dim, a)
    f = O.factors(r, rec)
    assert np.all(f[0][obs_dim:] == 0) and np.all(f[0][:obs_dim] != 0)
    assert np.all(f[5][a:] == 0) and np.all(f[5][:a] != 0)
    assert np.all(f[7][1:] == 0) and f[7][0] != 0
    assert np.all(r[rec.v_out + 4:] == 0)


class NoisyLinear(torch.nn.Module):
    """Fortunato et al.'s factorized NoisyLinear (y = x (mu_w + sigma_w * outer(f_in, f_out)) + mu_b + sigma_b * f_out)."""

    def __init__(self, mu_w, mu_b, sig_w, sig_b):
        super().__init__()
        self.mu_w, self.mu_b = torch.nn.Parameter(mu_w.clone()), torch.nn.Parameter(mu_b.clone())
        self.sig_w, self.sig_b = torch.nn.Parameter(sig_w.clone()), torch.nn.Parameter(sig_b.clone())

    def forward(self, x, f_in, f_out):
        return x @ (self.mu_w + self.sig_w * torch.outer(f_in, f_out)) + self.mu_b + self.sig_b * f_out


@pytest.mark.parametrize("dueling", [False, True])
def test_oracle_noisy_mlp_and_gradients_match_a_torch_nn_noisy_linear_network(dueling):
    from dmdqn_b200.group import keras_init
    torch.manual_seed(0)
    d, h, a, b = 89, 64, 4, 32
    rec = _rec(96, h)
    record = O.noise_record(99, 4, 0, rec, d, a)
    mu = keras_init(5, d, h, a, dueling)
    sg = [torch.rand_like(p) * 0.1 for p in mu]
    eps = O.eps_params(record, rec, d, a, dueling)
    orc = O.NoisyStackedOracle(1, d, [h, h], a, dueling=dueling)
    x = torch.randn(1, b, d)
    mu_p = [p[None].clone().requires_grad_(True) for p in mu]
    sg_p = [p[None].clone().requires_grad_(True) for p in sg]
    q = orc.forward(orc.effective(mu_p, sg_p, [e[None] for e in eps]), x)
    f = [torch.as_tensor(v) for v in O.factors(record, rec)]
    layers = [NoisyLinear(mu[2 * i], mu[2 * i + 1], sg[2 * i], sg[2 * i + 1]) for i in range(4 if dueling else 3)]
    h1 = torch.relu(layers[0](x[0], f[0][:d], f[1]))
    h2 = torch.relu(layers[1](h1, f[2], f[3]))
    qr = layers[2](h2, f[4], f[5][:a])
    if dueling:
        qr = layers[3](h2, f[6], f[7][:1]) + qr - qr.mean(dim=1, keepdim=True)
    torch.testing.assert_close(q[0], qr, rtol=1e-5, atol=1e-5)
    w = torch.randn(b, a)
    g = torch.autograd.grad((q[0] * w).sum(), mu_p + sg_p)
    (qr * w).sum().backward()
    ref = [p.grad for l in layers for p in (l.mu_w, l.mu_b)] + [p.grad for l in layers for p in (l.sig_w, l.sig_b)]
    for got, want in zip(g, ref):
        torch.testing.assert_close(got[0], want, rtol=1e-4, atol=1e-6)


def test_sigma_gradient_is_the_effective_gradient_times_eps_and_the_fold_is_one_product_and_one_sum():
    rng = np.random.default_rng(1)
    mu, sg, e = (rng.standard_normal(1000).astype(np.float32) for _ in range(3))
    eff = O.fold_np(mu, sg, e)
    assert np.array_equal(eff, np.float32(mu) + np.float32(sg * e))
    assert np.allclose(eff, mu.astype(np.float64) + sg.astype(np.float64) * e, rtol=1e-6, atol=1e-6)
    assert np.array_equal(O.fold_np(mu, np.zeros_like(sg), e), mu)           # sigma = 0: eff is mu bit for bit
    # W = mu + sigma * eps: dL/dmu = dL/dW, dL/dsigma = dL/dW * eps
    m, s = torch.tensor(mu, requires_grad=True), torch.tensor(sg, requires_grad=True)
    gw = torch.tensor(rng.standard_normal(1000).astype(np.float32))
    gm, gs = torch.autograd.grad(((m + s * torch.tensor(e)) * gw).sum(), (m, s))
    assert torch.equal(gm, gw) and torch.equal(gs, gw * torch.tensor(e))


def test_eps_block_places_every_layer_at_its_offsets():
    from dmdqn_b200.group import AgentGroup
    h, a = 64, 3
    rec = _rec(96, h)
    r = O.noise_record(3, 0, 0, rec, 89, a)
    L = SimpleNamespace(w1=0, b1=96 * h, w2=96 * h + h, b2=96 * h + h + h * h, w3=96 * h + 2 * h + h * h)
    L.b3 = L.w3 + 4 * h; L.wv = L.b3 + 4; L.bv = L.wv + h; L.stride = (L.bv + 4 + 31) // 32 * 32
    e = O.eps_block(r, rec, L, h, True)
    grp = SimpleNamespace(layout=L, hidden=h, action_size=a, obs_stride=96, state_size=89, dueling=True)
    blk = AgentGroup.pack(grp, O.eps_params(r, rec, 89, a, True)).numpy()
    assert np.array_equal(e[:L.bv + 1], blk[:L.bv + 1]) and np.all(e[L.bv + 1:] == 0)


@pytest.mark.parametrize("dueling", [False, True])
def test_sigma_init_is_sigma0_over_sqrt_fan_in_and_mu_is_keras_init(dueling):
    from dmdqn_b200.group import AgentGroup, keras_init
    grp = SimpleNamespace(state_size=89, hidden=64, action_size=4, dueling=dueling, noisy_sigma0=0.5)
    sig = AgentGroup.sigma_init(grp)
    want = [0.5 / math.sqrt(89)] * 2 + [0.5 / 8.0] * (6 if dueling else 4)
    assert [tuple(s.shape) for s in sig] == [tuple(p.shape) for p in keras_init(0, 89, 64, 4, dueling)]
    for s, w in zip(sig, want):
        assert torch.all(s == np.float32(w))


def test_noise_keys_depend_on_the_network_seed_alone():
    from dmdqn_b200.group import noise_key
    keys = [noise_key(s) for s in range(1000)]
    assert len(set(keys)) == 1000 and all(0 <= k < 1 << 64 for k in keys)
    assert noise_key(10 + 3) == noise_key(13)


def test_config_keys_default_off_and_in_the_yaml():
    from dmdqn_b200 import train
    from dmdqn_b200.group import DEFAULTS
    assert DEFAULTS["noisy"] is False and DEFAULTS["noisy_sigma0"] == 0.5
    cfg = train.load_config()
    assert cfg["noisy"] is False and cfg["noisy_sigma0"] == 0.5


@pytest.mark.parametrize("extra,match", [({"noisy": 1.0}, "noisy="), ({"noisy": "yes"}, "noisy="),
                                         ({"noisy": True, "noisy_sigma0": -0.1}, "noisy_sigma0"),
                                         ({"noisy": True, "noisy_sigma0": float("nan")}, "noisy_sigma0"),
                                         ({"noisy": True, "noisy_sigma0": "0.5"}, "noisy_sigma0"),
                                         ({"noisy": True, "global_clipnorm": 1.0}, "global_clipnorm")])
def test_agent_group_refuses_bad_noisy_config_before_loading_the_library(extra, match):
    from dmdqn_b200.group import AgentGroup
    with pytest.raises(ValueError, match=match):
        AgentGroup(4, {"nn_layers": [64, 64], **extra})


def test_fused_shared_step_with_noise_is_refused():
    class Shared:
        shared, global_clipnorm, noisy = True, None, True
    with pytest.raises(ValueError, match="sigma"):
        SharedParameterStep.for_group(Shared(), fused=True)


@pytest.fixture(scope="module")
def lib():
    from dmdqn_b200 import _native as N
    from dmdqn_b200 import build as B
    B.build()
    return N.lib()


def test_native_noise_layout(lib):
    from dmdqn_b200 import _native as N
    for h in (64, 128, 256, 512):
        dims = N.Dims(4, 4, 89, 96, h, 4, 32, 100)
        r = N.NoiseRecord()
        N.check(lib.dmdqn_noise_layout(C.byref(dims), C.byref(r)))
        want = _rec(96, h)
        assert all(getattr(r, k) == getattr(want, k) for k in ("w1_in", "w1_out", "w2_in", "w2_out", "w3_in", "w3_out",
                                                               "v_in", "v_out", "stride"))


def test_native_noisy_calls_refuse_null_and_misaligned_pointers_before_launching_anything(lib):
    from dmdqn_b200 import _native as N
    dims = N.Dims(4, 4, 89, 96, 64, 4, 32, 100)
    nbytes = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(dims), C.byref(nbytes)))
    ws = (C.c_uint8 * 256)()
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 1000, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100)
    rp = N.Replay(16, 16, 16, 16, 16, 16, None, None)
    nets = N.Nets(16, 16, 16, 16, 16)
    good = dict(zip(("sigma", "sigma_tgt", "sigma_m", "sigma_v", "eff", "eff_tgt", "noise", "key"), [16] * 8))
    err = lambda: lib.dmdqn_last_error().decode()

    def calls(nz, fold=True):
        if fold:                          # the fold does not touch the sigma moments
            yield lib.dmdqn_noisy_fold(C.byref(dims), C.byref(hp), C.byref(nets), C.byref(nz), None)
        yield lib.dmdqn_learn_grads_noisy(C.byref(dims), C.byref(hp), C.byref(rp), C.byref(nets), C.byref(nz), 16, None, 32, 16,
                                          16, C.addressof(ws), nbytes.value, None)
        yield lib.dmdqn_noisy_adam_apply(C.byref(dims), C.byref(hp), C.byref(nets), C.byref(nz), 16, C.addressof(ws),
                                         nbytes.value, None)
    for k in good:
        for rc in calls(N.Noisy(**dict(good, **{k: None})), fold=k not in ("sigma_m", "sigma_v")):
            assert rc == N.ERR_ARG and "NULL" in err(), k
    for rc in calls(N.Noisy(**dict(good, eff=20))):
        assert rc == N.ERR_ARG and "aligned" in err()
    assert lib.dmdqn_act_noisy(C.byref(dims), C.byref(nets), C.byref(N.Noisy(**dict(good, sigma=None))), 0, 16, 96, 16, 16, 16,
                               16, None, None) == N.ERR_ARG
    assert lib.dmdqn_act_noisy(C.byref(dims), C.byref(nets), C.byref(N.Noisy(**good)), 2, 16, 96, 16, 16, 16, 16, None,
                               None) == N.ERR_ARG
    assert lib.dmdqn_sync_target_noisy(C.byref(dims), C.byref(nets), C.byref(N.Noisy(**dict(good, sigma_tgt=None))), 0, None,
                                       -1.0, None) == N.ERR_ARG
    assert lib.dmdqn_learn_grads_noisy(C.byref(dims), C.byref(hp), C.byref(rp), C.byref(nets), C.byref(N.Noisy(**good)), 16,
                                       None, 32, 16, 16, C.addressof(ws), nbytes.value - 1, None) == N.ERR_WORKSPACE


# ------------------------------------------------------------------ gloo, world size 2 ----------------------------------
H, B_GLOBAL, KEY = 64, 64, 0x0123_4567_89ab_cdef


def _data():
    rng = np.random.default_rng(0)
    S = rng.integers(-1, 20, (1, B_GLOBAL, 89)).astype(np.float32)
    S2 = rng.integers(-1, 20, (1, B_GLOBAL, 89)).astype(np.float32)
    A_ = rng.integers(0, 4, (1, B_GLOBAL)); R = (rng.standard_normal((1, B_GLOBAL)) * 20).astype(np.float32)
    D = (rng.random((1, B_GLOBAL)) < 0.1).astype(np.float32)
    return S, A_, R, S2, D


def _eps(t, s):
    rec = _rec(96, H)
    return [e[None] for e in O.eps_params(O.noise_record(KEY, t, s, rec, 89, 4), rec, 89, 4, False)]


def _oracle():
    orc = O.NoisyStackedOracle(1, 89, [H, H], 4, seed0=3)
    orc.sigma = [torch.full_like(p, 0.05) for p in orc.online]
    orc.sigma_tgt = [p.clone() for p in orc.sigma]
    orc.sigma_m = [torch.zeros_like(p) for p in orc.online]
    orc.sigma_v = [torch.zeros_like(p) for p in orc.online]
    return orc


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from oracle.dqn import adam_scalars, adam_update_, loss_and_grad
        torch.set_num_threads(1)
        b_local = B_GLOBAL // world
        S, A_, R, S2, D = _data()
        sl = slice(rank * b_local, (rank + 1) * b_local)
        orc = _oracle()

        def local_grads(global_batch):     # dmdqn_learn_grads_noisy: the gradient of the effective weights
            t = int(orc.learn_step[0])
            e_on, e_tg = _eps(t, 0), _eps(t, 1)
            with torch.no_grad():
                tq_all = orc.forward(orc.effective(orc.target, orc.sigma_tgt, e_tg), torch.as_tensor(S2[:, sl]))
                q_next = orc.forward(orc.effective(orc.online, orc.sigma, e_on), torch.as_tensor(S2[:, sl]))
                tq = torch.gather(tq_all, 2, torch.argmax(q_next, dim=2, keepdim=True))[..., 0]
                y = torch.as_tensor(R[:, sl]) + np.float32(orc.gamma) * (1 - torch.as_tensor(D[:, sl])) * tq
            eff = [w.detach().requires_grad_(True) for w in orc.effective(orc.online, orc.sigma, e_on)]
            pred = torch.gather(orc.forward(eff, torch.as_tensor(S[:, sl])), 2, torch.as_tensor(A_[:, sl])[..., None])[..., 0]
            terms, _ = loss_and_grad(pred, y, "mse")
            loss = terms.sum(dim=1) / global_batch
            grads = torch.autograd.grad(loss.sum(), eff)
            metrics = torch.zeros(1, 8); metrics[0, 0] = loss.detach()[0]
            return torch.cat([g.reshape(-1) for g in grads]), metrics

        def apply(flat):                  # dmdqn_noisy_adam_apply on the all-reduced block
            e_on = _eps(int(orc.learn_step[0]), 0)
            orc.learn_step[0] += 1
            alpha, eps = adam_scalars(int(orc.learn_step[0]), orc.lr)
            off = 0
            with torch.no_grad():
                for k in range(len(orc.online)):
                    n = orc.online[k].numel()
                    g = flat[off:off + n].view_as(orc.online[k])
                    adam_update_(orc.online[k], g, orc.adam_m[k], orc.adam_v[k], alpha, eps)
                    adam_update_(orc.sigma[k], g * e_on[k], orc.sigma_m[k], orc.sigma_v[k], alpha, eps)
                    off += n

        step = SharedParameterStep(local_grads, apply, b_local)
        for _ in range(2):
            step.step()
        q.put((rank, [p.clone().numpy() for p in orc.online + orc.sigma]))
    finally:
        dist.destroy_process_group()


def test_shared_parameter_noisy_step_equals_single_process_big_batch_noisy_step():
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
    ref = _oracle()
    for _ in range(2):
        t = int(ref.learn_step[0])
        ref.learn_on_batch(S, A_, R, S2, D, _eps(t, 0), _eps(t, 1))
    for rank, weights in results:
        for w, r in zip(weights, ref.online + ref.sigma):
            np.testing.assert_allclose(w, r.numpy(), rtol=1e-5, atol=1e-6)
    for w0, w1 in zip(results[0][1], results[1][1]):    # the same noise and the same block on every rank
        assert np.array_equal(w0, w1)
