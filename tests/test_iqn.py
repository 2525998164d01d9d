"""CPU checks of implicit quantile networks (IQN): the fractions, the cosine features, the oracle's forward pass, loss and
gradients against independent float64 torch code, the host-side configuration and the C ABI's exports and refusals (no GPU
needed: every refusal happens before a launch)."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

import iqn_oracle as IO
import quantile_oracle as QO
from dmdqn_b200 import _native as N
from dmdqn_b200 import build as B
from dmdqn_b200.group import DEFAULTS, dist_config, iqn_config, keras_init, noise_key, quantile_config


@pytest.fixture(scope="module")
def lib():
    B.build()
    return N.lib()


# ------------------------------------------------------------------ fractions and features ------------------------------
def test_fractions_lie_on_the_23_bit_grid_strictly_inside_the_unit_interval():
    key = noise_key(5)
    tau = IO.fractions(key, np.arange(512), 64, 3, 0)
    k = tau.astype(np.float64) * 2.0 ** 23 - 0.5
    assert np.array_equal(k, np.round(k)) and np.all(tau > 0) and np.all(tau < 1)
    assert tau.dtype == np.float32 and abs(float(tau.mean()) - 0.5) < 0.01
    edge = ((np.array([0, 2 ** 23 - 1], np.uint32)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -23)
    assert edge[0] == 2.0 ** -24 and edge[1] == 1 - 2.0 ** -24           # the extremes are exact and inside (0, 1)


def test_fractions_are_keyed_by_every_counter_field():
    key = noise_key(1)
    base = IO.fractions(key, np.arange(16), 8, 4, 0)
    others = [IO.fractions(noise_key(2), np.arange(16), 8, 4, 0), IO.fractions(key, np.arange(16) + 16, 8, 4, 0),
              IO.fractions(key, np.arange(16), 8, 5, 0), IO.fractions(key, np.arange(16), 8, 4, 1)]
    for o in others:
        assert np.mean(o == base) < 0.01
    assert np.array_equal(IO.fractions(key, np.arange(16), 16, 4, 0)[:, :8], base)        # fraction i is its own counter
    assert np.array_equal(IO.fractions(key, np.arange(4, 12), 8, 4, 0), base[4:12])     # row r is its own counter


def test_cosine_features_are_within_one_ulp_of_float64():
    tau = IO.fractions(noise_key(3), np.arange(64), 8, 0, 0)
    c = IO.cos_features(tau, 128)
    ref = np.cos(np.pi * np.arange(128) * tau.astype(np.float64)[..., None])
    ulp = np.spacing(np.abs(c)).astype(np.float64)
    assert np.all(np.abs(c - ref) <= ulp) and c.dtype == np.float32
    assert np.all(c[..., 0] == 1)


# ------------------------------------------------------------------ the model -------------------------------------------
class TorchIQN(torch.nn.Module):
    """IQN as Dabney et al. (2018) build it, in torch.nn and float64: psi = relu(Linear(s)), phi = relu(Linear(cos(pi i tau))),
    f = Linear(relu(Linear(psi * phi)))."""

    def __init__(self, d, h, a, n_cos):
        super().__init__()
        self.n_cos = n_cos
        self.psi, self.phi = torch.nn.Linear(d, h).double(), torch.nn.Linear(n_cos, h).double()
        self.f1, self.f2 = torch.nn.Linear(h, h).double(), torch.nn.Linear(h, a).double()

    def load(self, w):          # [W1, b1, W2, b2, W3, b3, Wphi, bphi] of one network, kernels [in, out]
        with torch.no_grad():
            for mod, (k, b) in ((self.psi, w[0:2]), (self.f1, w[2:4]), (self.f2, w[4:6]), (self.phi, w[6:8])):
                mod.weight.copy_(torch.as_tensor(np.asarray(k)).double().T)
                mod.bias.copy_(torch.as_tensor(np.asarray(b)).double())
        return self

    def params(self):
        return [self.psi.weight, self.psi.bias, self.f1.weight, self.f1.bias, self.f2.weight, self.f2.bias, self.phi.weight,
                self.phi.bias]

    def forward(self, s, tau):  # s [B, D], tau [B, M] -> [B, M, A]
        i = torch.arange(self.n_cos, dtype=torch.float64)
        emb = torch.relu(self.phi(torch.cos(math.pi * i * tau[..., None])))
        return self.f2(torch.relu(self.f1(torch.relu(self.psi(s))[:, None] * emb)))


def paper_loss(theta, t, tau, kappa):
    """Per-row loss: sum over i of the mean over j of |tau_i - 1{u < 0}| L_kappa(u) / kappa (kappa > 0) or
    |tau_i - 1{u < 0}| |u| (kappa = 0), u = T_j - theta_i."""
    u = t[..., None, :] - theta[..., :, None]
    w = (tau[..., :, None] - (u < 0).double()).abs()
    if kappa > 0:
        rho = w * torch.where(u.abs() <= kappa, 0.5 * u * u, kappa * (u.abs() - 0.5 * kappa)) / kappa
    else:
        rho = w * u.abs()
    return rho.mean(-1).sum(-1)


def _batch(rng, g, b, d, a):
    s = rng.integers(-1, 20, (g, b, d)).astype(np.float32)
    s2 = rng.integers(-1, 20, (g, b, d)).astype(np.float32)
    return (s, rng.integers(0, a, (g, b)), rng.uniform(-3, 3, (g, b)).astype(np.float32), s2,
            rng.choice([0.0, 0.99], (g, b)).astype(np.float32))


def test_forward_matches_a_torch_nn_module():
    rng = np.random.default_rng(1)
    o = IO.IqnOracle(2, 89, 64, 3, n_cos=16, seed0=4)
    s = rng.integers(-1, 20, (2, 8, 89)).astype(np.float32)
    tau = np.stack([IO.fractions(noise_key(4 + g), np.arange(8), 5, 0, 0) for g in range(2)])
    with torch.no_grad():
        z = IO.forward(o.online, s, tau).numpy()
    for g in range(2):
        m = TorchIQN(89, 64, 3, 16).load([p[g] for p in o.online])
        ref = m(torch.as_tensor(s[g]).double(), torch.as_tensor(tau[g]).double()).detach().numpy()
        assert np.abs(z[g] - ref).max() < 1e-5 * max(1.0, np.abs(ref).max())


def test_initial_weights_extend_keras_init_after_every_plain_weight():
    w = keras_init(7, 89, 64, 4, n_cos=32)
    assert [tuple(x.shape) for x in w] == [(89, 64), (64,), (64, 64), (64,), (64, 4), (4,), (32, 64), (64,)]
    for x, y in zip(w[:6], keras_init(7, 89, 64, 4)):
        assert torch.equal(x, y)
    for x, y in zip(w, IO.init_params(7, 89, 64, 4, 32)):
        assert torch.equal(x, y)
    std = math.sqrt(2.0 / 32) / 0.87962566103423978
    assert float(w[6].abs().max()) <= 2 * std and torch.all(w[7] == 0)


@pytest.mark.parametrize("kappa", [1.0, 0.0])
@pytest.mark.parametrize("n,n_p", [(8, 8), (13, 5), (1, 1)])
def test_closed_form_gradient_matches_float64_autograd(kappa, n, n_p):
    rng = np.random.default_rng(n * 7 + n_p)
    theta = rng.standard_normal((64, n)).astype(np.float32) * 2
    t = rng.standard_normal((64, n_p)).astype(np.float32) * 2
    tau = IO.fractions(noise_key(n), np.arange(64), n, 1, 0)
    L, g = IO.row_loss_and_grad(theta, t, tau, kappa)
    th64 = torch.as_tensor(theta, dtype=torch.float64).requires_grad_(True)
    ref = paper_loss(th64, torch.as_tensor(t, dtype=torch.float64), torch.as_tensor(tau, dtype=torch.float64), kappa)
    gref = torch.autograd.grad(ref.sum(), th64)[0].numpy()
    assert np.abs(g - gref).max() < 1e-6 * max(1.0, np.abs(gref).max())
    r = ref.detach().numpy()
    assert np.abs(L - r).max() < 1e-5 * max(1.0, np.abs(r).max())


@pytest.mark.parametrize("kappa", [1.0, 0.0])
@pytest.mark.parametrize("n", [2, 8, 50])
def test_midpoint_fractions_give_qr_dqn_bit_for_bit(kappa, n):
    rng = np.random.default_rng(n)
    theta = rng.standard_normal((32, n)).astype(np.float32)
    t = rng.standard_normal((32, n)).astype(np.float32)
    L, g = IO.row_loss_and_grad(theta, t, np.broadcast_to(QO.midpoints(n), (32, n)), kappa)
    Lq, gq = QO.row_loss_and_grad(theta, t, kappa)
    assert np.array_equal(L, Lq) and np.array_equal(g, gq)


def test_oracle_parameter_gradients_match_float64_autograd():
    rng = np.random.default_rng(7)
    g_, b, d, h, a, n_cos, kappa = 2, 16, 89, 64, 3, 16, 1.0
    o = IO.IqnOracle(g_, d, h, a, n_cos=n_cos, n_tau=6, n_tau_prime=5, n_policy=7, kappa=kappa, seed0=3)
    s, act, r, s2, disc = _batch(rng, g_, b, d, a)
    w = rng.uniform(0.2, 1.0, (g_, b)).astype(np.float32)
    tau = np.stack([IO.fractions(noise_key(3 + g), np.arange(b), 6, 0, 0) for g in range(g_)])
    tau_p = np.stack([IO.fractions(noise_key(3 + g), np.arange(b), 5, 0, 1) for g in range(g_)])
    out = o.learn_on_batch(s, act, r, s2, disc, tau, tau_p, is_weights=w, apply=False)
    for g in range(g_):
        m = TorchIQN(d, h, a, n_cos).load([p[g] for p in o.online])
        z = m(torch.as_tensor(s[g]).double(), torch.as_tensor(tau[g]).double())
        th = torch.gather(z, 2, torch.as_tensor(act[g])[:, None, None].expand(b, 6, 1))[..., 0]
        row = paper_loss(th, torch.as_tensor(out["T"][g]).double(), torch.as_tensor(tau[g]).double(), kappa)
        loss = (torch.as_tensor(w[g]).double() * row).mean()
        grads = torch.autograd.grad(loss, m.params())
        mine = out["grads"]
        for k, ref in enumerate(grads):
            ref = ref.numpy().T if ref.dim() == 2 else ref.numpy()
            assert np.abs(mine[k][g] - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), k
        ref = float(loss.detach())
        assert abs(out["loss"][g] - ref) < 1e-5 * max(1.0, abs(ref))


def test_a_few_oracle_steps_match_an_independent_float64_learner():
    rng = np.random.default_rng(11)
    g_, b, d, h, a, n_cos, kappa, lr = 1, 32, 89, 64, 4, 16, 1.0, 1e-3
    o = IO.IqnOracle(g_, d, h, a, n_cos=n_cos, n_tau=8, n_tau_prime=8, n_policy=8, kappa=kappa, learning_rate=lr, seed0=9,
                     target_update_frequency=1000)
    on = TorchIQN(d, h, a, n_cos).load([p[0] for p in o.online])
    tg = TorchIQN(d, h, a, n_cos).load([p[0] for p in o.online])
    ms = [torch.zeros_like(p) for p in on.params()]
    vs = [torch.zeros_like(p) for p in on.params()]
    mid = torch.as_tensor(QO.midpoints(8)).double()
    for step in range(3):
        s, act, r, s2, disc = _batch(rng, g_, b, d, a)
        tau = IO.fractions(noise_key(9), np.arange(b), 8, step, 0)[None]
        tau_p = IO.fractions(noise_key(9), np.arange(b), 8, step, 1)[None]
        o.learn_on_batch(s, act, r, s2, disc, tau, tau_p)
        with torch.no_grad():
            s2t = torch.as_tensor(s2[0]).double()
            best = on(s2t, mid.expand(b, 8)).mean(1).argmax(1)
            zt = tg(s2t, torch.as_tensor(tau_p[0]).double())
            t = torch.as_tensor(r[0]).double()[:, None] + torch.as_tensor(disc[0]).double()[:, None] * \
                torch.gather(zt, 2, best[:, None, None].expand(b, 8, 1))[..., 0]
        z = on(torch.as_tensor(s[0]).double(), torch.as_tensor(tau[0]).double())
        th = torch.gather(z, 2, torch.as_tensor(act[0])[:, None, None].expand(b, 8, 1))[..., 0]
        loss = paper_loss(th, t, torch.as_tensor(tau[0]).double(), kappa).mean()
        grads = torch.autograd.grad(loss, on.params())
        alpha, eps = 1e-3 * math.sqrt(1 - 0.999 ** (step + 1)) / (1 - 0.9 ** (step + 1)), 1e-7
        with torch.no_grad():
            for p, gg, m_, v_ in zip(on.params(), grads, ms, vs):
                m_ += (gg - m_) * 0.1
                v_ += (gg * gg - v_) * 0.001
                p -= (m_ * alpha) / (v_.sqrt() + eps)
        for k, p in enumerate(on.params()):
            ref = p.detach().numpy().T if p.dim() == 2 else p.detach().numpy()
            assert np.abs(o.online[k][0].numpy() - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max()), (step, k)


# ------------------------------------------------------------------ C ABI (no GPU) -------------------------------------
def test_exports(lib):
    for name in ("dmdqn_param_layout_iqn", "dmdqn_iqn_scratch_bytes", "dmdqn_learn_grads_iqn", "dmdqn_adam_apply_iqn",
                 "dmdqn_act_iqn", "dmdqn_sync_target_iqn", "dmdqn_debug_iqn"):
        assert name in N.SIGNATURES and hasattr(lib, name)
    assert C.sizeof(N.Iqn) == 56 and C.sizeof(N.IqnLayout) == 80 and C.sizeof(N.IqnViews) == 56 and lib.dmdqn_abi_version() == 3


@pytest.mark.parametrize("h,n_cos", [(64, 4), (256, 64), (512, 128)])
def test_layout(lib, h, n_cos):
    d = N.Dims(2, 2, 89, 96, h, 4, 32, 100)
    L, P = N.IqnLayout(), N.Layout()
    N.check(lib.dmdqn_param_layout_iqn(C.byref(d), n_cos, C.byref(L)))
    N.check(lib.dmdqn_param_layout(C.byref(d), C.byref(P)))
    assert (L.w1, L.b1, L.w2, L.b2, L.w3, L.b3) == (P.w1, P.b1, P.w2, P.b2, P.w3, P.b3)
    assert L.wphi == L.b3 + 4 and L.wphi % 4 == 0 and L.bphi == L.wphi + n_cos * h and L.end == L.bphi + h
    assert L.stride % 32 == 0 and L.end <= L.stride < L.end + 32


def test_scratch_query(lib):
    d = N.Dims(3, 3, 89, 96, 128, 4, 40, 100)
    q = N.Iqn(8, 5, 32, 64, 1.0, 0, None, None, 0)
    nb = C.c_size_t()
    N.check(lib.dmdqn_iqn_scratch_bytes(C.byref(d), C.byref(q), C.byref(nb)))
    up = lambda x: (x + 255) // 256 * 256
    rows = 3 * 40
    want = up(rows * 8 * 4) + 2 * up(rows * 5 * 4) + 2 * up(rows * 8 * 4) + up(2 * rows * 128 * 4) + up(rows * 8 * 64 * 4) + \
        3 * up(rows * 8 * 128 * 4) + up(3 * 1 * 128 * 4)
    assert nb.value == want
    buf = (C.c_char * (want + 256))()
    base = (C.addressof(buf) + 255) // 256 * 256
    q.scratch, q.scratch_bytes = base, want
    v = N.IqnViews()
    N.check(lib.dmdqn_debug_iqn(C.byref(d), C.byref(q), C.byref(v)))
    assert v.tau == base and v.tau_prime == base + up(rows * 8 * 4) and v.target == v.tau_prime + up(rows * 5 * 4)
    assert v.theta == v.target + up(rows * 5 * 4) and v.grad == v.theta + up(rows * 8 * 4)
    h2 = v.grad + up(rows * 8 * 4) + up(2 * rows * 128 * 4) + up(rows * 8 * 64 * 4) + up(rows * 8 * 128 * 4)
    assert v.dh2 == h2 and v.dphi == h2 + up(rows * 8 * 128 * 4)


def _buf(n=1 << 16):
    raw = (C.c_char * (n + 256))()
    return raw, (C.addressof(raw) + 255) // 256 * 256


CASES = {"n0": "n_tau", "n65": "n_tau", "np0": "n_tau_prime", "k65": "n_policy", "cos2": "n_cos", "cos6": "n_cos",
         "cos132": "n_cos", "kappa_neg": "kappa", "kappa_nan": "kappa", "kappa_inf": "kappa", "row_base": "row_base",
         "tf32x3": "precision", "dueling": "dueling", "null_key": "key", "small_scratch": "scratch", "null_scratch": "scratch",
         "misaligned_scratch": "scratch", "misaligned_grads": "grads_out", "null_iqn": "iqn"}


@pytest.mark.parametrize("case", list(CASES))
def test_abi_refusals(lib, case):
    d = N.Dims(2, 2, 89, 96, 64, 4, 32, 100)
    keep, base = _buf(1 << 22)
    ws = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(d), C.byref(ws)))
    ws_keep, ws_ptr = _buf(ws.value)
    q = N.Iqn(8, 8, 32, 64, 1.0, 0, base, None, 0)
    sb = C.c_size_t()
    N.check(lib.dmdqn_iqn_scratch_bytes(C.byref(d), C.byref(q), C.byref(sb)))
    sc_keep, sc_ptr = _buf(sb.value)
    q.scratch, q.scratch_bytes = sc_ptr, sb.value
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 10, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100, 1)
    nets = N.Nets(base, base + 4096, base + 8192, base + 12288, base + 16384)
    replay = N.Replay(base, base, base, base, base, base, None, None)
    grads = base + 65536
    edits = {"n0": ("n_tau", 0), "n65": ("n_tau", 65), "np0": ("n_tau_prime", 0), "k65": ("n_policy", 65), "cos2": ("n_cos", 2),
             "cos6": ("n_cos", 6), "cos132": ("n_cos", 132), "kappa_neg": ("kappa", -0.5), "kappa_nan": ("kappa", float("nan")),
             "kappa_inf": ("kappa", float("inf")), "row_base": ("row_base", -1), "null_key": ("key", None),
             "small_scratch": ("scratch_bytes", sb.value - 1), "null_scratch": ("scratch", None),
             "misaligned_scratch": ("scratch", sc_ptr + 4)}
    if case in edits:
        setattr(q, *edits[case])
    elif case == "tf32x3":
        hp.precision = 2
    elif case == "dueling":
        hp.dueling = 1
    elif case == "misaligned_grads":
        grads += 4
    qp = None if case == "null_iqn" else C.byref(q)
    rc = lib.dmdqn_learn_grads_iqn(C.byref(d), C.byref(hp), qp, C.byref(replay), C.byref(nets), base, None, 32, grads, None,
                                   ws_ptr, ws.value, None)
    assert rc == N.ERR_ARG
    assert CASES[case] in lib.dmdqn_last_error().decode()
    if case in ("n0", "n65", "np0", "k65", "cos2", "cos6", "cos132", "kappa_neg", "kappa_nan", "kappa_inf", "row_base",
                "null_iqn"):
        assert lib.dmdqn_act_iqn(C.byref(d), C.byref(nets), qp, base, 96, base, base, base, base, None, None) == N.ERR_ARG
        assert lib.dmdqn_debug_iqn(C.byref(d), qp, C.byref(N.IqnViews())) == N.ERR_ARG
    if case.startswith("cos"):
        assert lib.dmdqn_param_layout_iqn(C.byref(d), q.n_cos, C.byref(N.IqnLayout())) == N.ERR_ARG
        assert lib.dmdqn_sync_target_iqn(C.byref(d), C.byref(nets), q.n_cos, None, -1.0, None) == N.ERR_ARG
        assert lib.dmdqn_adam_apply_iqn(C.byref(d), C.byref(hp), C.byref(nets), q.n_cos, grads, 0.0, None, ws_ptr, ws.value,
                                        None) == N.ERR_ARG
    if case in ("tf32x3", "dueling"):
        assert lib.dmdqn_adam_apply_iqn(C.byref(d), C.byref(hp), C.byref(nets), 64, grads, 0.0, None, ws_ptr, ws.value,
                                        None) == N.ERR_ARG


def test_adam_apply_refuses_a_bad_clipnorm(lib):
    d = N.Dims(2, 2, 89, 96, 64, 4, 32, 100)
    keep, base = _buf(1 << 20)
    ws = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(d), C.byref(ws)))
    ws_keep, ws_ptr = _buf(ws.value)
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 10, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100, 1)
    nets = N.Nets(base, base + 4096, base + 8192, base + 12288, base + 16384)
    for c in (-1.0, float("nan"), float("inf")):
        assert lib.dmdqn_adam_apply_iqn(C.byref(d), C.byref(hp), C.byref(nets), 64, base, c, None, ws_ptr, ws.value,
                                        None) == N.ERR_ARG
        assert "global_clipnorm" in lib.dmdqn_last_error().decode()


# ------------------------------------------------------------------ host configuration ---------------------------------
def _cfg(**kw):
    cfg = dict(DEFAULTS, iqn=True)
    cfg.update(kw)
    return cfg


def test_auto_precision_resolves_to_fp32_and_other_configs_are_untouched():
    assert iqn_config(_cfg())["precision"] == "fp32"
    assert iqn_config(_cfg(precision="fp32", quantile_kappa=0))["precision"] == "fp32"
    plain = dict(DEFAULTS)
    assert iqn_config(dict(plain)) == plain
    assert dist_config(_cfg()) == _cfg() and quantile_config(_cfg()) == _cfg()


@pytest.mark.parametrize("kw,word", [({"precision": "tf32x3"}, "precision"), ({"precision": "tf32"}, "precision"),
                                     ({"distributional": True}, "distributional"), ({"quantile": True}, "quantile"),
                                     ({"dueling": True}, "dueling"), ({"noisy": True}, "noisy"), ({"loss": "huber"}, "loss"),
                                     ({"iqn_num_tau": 0}, "iqn_num_tau"), ({"iqn_num_tau": 65}, "iqn_num_tau"),
                                     ({"iqn_num_tau_prime": 0}, "iqn_num_tau_prime"),
                                     ({"iqn_num_policy_tau": 65}, "iqn_num_policy_tau"),
                                     ({"iqn_num_tau": 8.0}, "iqn_num_tau"), ({"iqn_num_tau": True}, "iqn_num_tau"),
                                     ({"iqn_embedding_dim": 6}, "iqn_embedding_dim"),
                                     ({"iqn_embedding_dim": 132}, "iqn_embedding_dim"),
                                     ({"iqn_embedding_dim": 0}, "iqn_embedding_dim"),
                                     ({"quantile_kappa": -1.0}, "quantile_kappa"),
                                     ({"quantile_kappa": float("nan")}, "quantile_kappa"), ({"iqn": "yes"}, "iqn")])
def test_host_refusals(kw, word):
    with pytest.raises(ValueError, match=word):
        iqn_config(_cfg(**kw))


def test_defaults_and_config_yaml_have_the_keys():
    import yaml
    want = {"iqn": False, "iqn_num_tau": 8, "iqn_num_tau_prime": 8, "iqn_num_policy_tau": 32, "iqn_embedding_dim": 64}
    path = os.path.join(os.path.dirname(__file__), "..", "config", "agent_config.yaml")
    cfg = yaml.safe_load(open(path))
    for k, v in want.items():
        assert DEFAULTS[k] == v and cfg[k] == v and type(cfg[k]) is type(v), k
