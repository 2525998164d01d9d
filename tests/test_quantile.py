"""CPU checks of quantile regression DQN (QR-DQN): the oracle's loss and gradients, the host-side configuration and the C
ABI's exports and refusals (no GPU needed: every refusal happens before a launch)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import quantile_oracle as QO
from dmdqn_b200 import _native as N
from dmdqn_b200 import build as B
from dmdqn_b200.group import DEFAULTS, dist_config, quantile_config


@pytest.fixture(scope="module")
def lib():
    B.build()
    return N.lib()


def _loss64(theta, t, kappa, n):
    """The per-row loss in float64 torch, as Dabney et al. (2018) write it: sum over i of the mean over j of
    |tau_i - 1{u < 0}| L_kappa(u) / kappa (kappa > 0) or |tau_i - 1{u < 0}| |u| (kappa = 0), u = T_j - theta_i."""
    tau = (2 * torch.arange(n, dtype=torch.float64) + 1) / (2 * n)
    u = t[..., None, :] - theta[..., :, None]
    w = (tau[:, None] - (u < 0).double()).abs()
    if kappa > 0:
        hub = torch.where(u.abs() <= kappa, 0.5 * u * u, kappa * (u.abs() - 0.5 * kappa))
        rho = w * hub / kappa
    else:
        rho = w * u.abs()
    return rho.mean(-1).sum(-1)


# ------------------------------------------------------------------ loss and gradients ---------------------------------
@pytest.mark.parametrize("kappa", [1.0, 0.5, 0.0])
@pytest.mark.parametrize("n", [2, 11, 50])
def test_closed_form_gradient_matches_float64_autograd(kappa, n):
    rng = np.random.default_rng(int(kappa * 10) + n)
    theta = rng.standard_normal((64, n)).astype(np.float32) * 2
    t = rng.standard_normal((64, n)).astype(np.float32) * 2
    L, g = QO.row_loss_and_grad(theta, t, kappa)
    th64 = torch.as_tensor(theta, dtype=torch.float64).requires_grad_(True)
    ref = _loss64(th64, torch.as_tensor(t, dtype=torch.float64), kappa, n)
    gref = torch.autograd.grad(ref.sum(), th64)[0].numpy()
    assert np.abs(g - gref).max() < 1e-6 * max(1.0, np.abs(gref).max())
    r = ref.detach().numpy()
    assert np.abs(L - r).max() < 1e-5 * max(1.0, np.abs(r).max())


def test_loss_is_zero_at_the_targets_only_for_equal_samples_and_grows_away():
    t = np.full((1, 4), 1.5, np.float32)
    L, g = QO.row_loss_and_grad(t.copy(), t, 1.0)
    assert L[0] == 0 and np.all(g == 0)
    L2, g2 = QO.row_loss_and_grad(t - 1, t, 1.0)     # every quantile below every sample: pushed up (g < 0)
    assert L2[0] > 0 and np.all(g2 < 0)


def test_midpoints():
    assert np.array_equal(QO.midpoints(2), np.array([0.25, 0.75], np.float32))
    tau = QO.midpoints(50)
    assert tau[0] == np.float32(0.01) and tau[-1] == np.float32(0.99) and np.all(np.diff(tau) > 0)


def test_oracle_parameter_gradients_match_autograd():
    """The oracle's logit gradient and its W / b gradients against float64 autograd of mean_r w_r L_r."""
    rng = np.random.default_rng(7)
    n_q, a, b, d, h, kappa = 11, 3, 16, 89, 64, 1.0
    o = QO.QuantileOracle(2, d, [h, h], a, n_q, kappa, seed0=3)
    for k in (1, 3, 5):
        o.online[k] += torch.as_tensor(rng.standard_normal(o.online[k].shape).astype(np.float32)) * 0.05
    o.target = [p.clone() for p in o.online]
    s = rng.integers(-1, 20, (2, b, d)).astype(np.float32)
    s2 = rng.integers(-1, 20, (2, b, d)).astype(np.float32)
    act = rng.integers(0, a, (2, b))
    r = rng.uniform(-3, 3, (2, b)).astype(np.float32)
    disc = rng.choice([0.0, 0.99], (2, b)).astype(np.float32)
    w = rng.uniform(0.2, 1.0, (2, b)).astype(np.float32)
    out = o.learn_on_batch(s, act, r, s2, None, is_weights=w, discounts=disc, apply=False)
    t = torch.as_tensor(out["T"], dtype=torch.float64)
    params = [p.detach().double().requires_grad_(True) for p in o.online]
    x = o.forward(params, torch.as_tensor(s, dtype=torch.float64)).reshape(2, b, a, n_q)
    xa = torch.gather(x, 2, torch.as_tensor(act)[..., None, None].expand(2, b, 1, n_q))[:, :, 0]
    row = _loss64(xa, t, kappa, n_q)
    loss = (torch.as_tensor(w, dtype=torch.float64) * row).mean(1).sum()
    gx = torch.autograd.grad(loss, [x], retain_graph=True)[0]
    assert np.abs(out["dlogits"] - gx.reshape(2, b, a, n_q).numpy()).max() < 1e-7
    grads = torch.autograd.grad(loss, params)
    for k, (g, ref) in enumerate(zip(out["grads"], grads)):
        assert np.abs(g - ref.numpy()).max() <= 1e-6 * max(1.0, float(ref.abs().max())), k
    ref_row = row.detach().numpy()
    assert np.abs(out["row_loss"] - ref_row).max() < 1e-6 * np.abs(ref_row).max()


def test_targets_follow_the_double_dqn_action():
    rng = np.random.default_rng(2)
    o = QO.QuantileOracle(1, 89, [64, 64], 4, 5, 1.0, seed0=1)
    s2 = rng.integers(-1, 20, (1, 8, 89)).astype(np.float32)
    r = rng.uniform(-1, 1, (1, 8)).astype(np.float32)
    d = np.full((1, 8), 0.99, np.float32)
    t, best, q_next, _ = o.targets(r, s2, d)
    assert np.array_equal(best, q_next.argmax(2))
    with torch.no_grad():
        xt = o.quantiles(o.target, s2).numpy()
    th = np.take_along_axis(xt, best[..., None, None], 2)[:, :, 0]
    assert np.array_equal(t, (r[..., None] + (d[..., None] * th).astype(np.float32)).astype(np.float32))


# ------------------------------------------------------------------ C ABI (no GPU) -------------------------------------
def test_exports(lib):
    for name in ("dmdqn_learn_grads_quantile", "dmdqn_act_quantile", "dmdqn_debug_quantile"):
        assert name in N.SIGNATURES and hasattr(lib, name)
    assert C.sizeof(N.Quantile) == 32


def _buf(n=1 << 16):
    raw = (C.c_char * (n + 256))()
    return raw, (C.addressof(raw) + 255) // 256 * 256


@pytest.mark.parametrize("case", ["n1", "n65", "kappa_neg", "kappa_nan", "kappa_inf", "tf32x3", "dueling", "small_scratch",
                                  "null_scratch", "misaligned_grads", "null_quantile"])
def test_abi_refusals(lib, case):
    d = N.Dims(2, 2, 89, 96, 64, 4, 32, 100)
    keep, base = _buf(1 << 22)
    ws = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(d), C.byref(ws)))
    ws_keep, ws_ptr = _buf(ws.value)
    sb = C.c_size_t()
    N.check(lib.dmdqn_dist_scratch_bytes(C.byref(d), 11, C.byref(sb)))
    sc_keep, sc_ptr = _buf(sb.value)
    qr = N.Quantile(11, 1.0, sc_ptr, sb.value)
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 10, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100, 1)
    nets = N.Nets(base, base + 4096, base + 8192, base + 12288, base + 16384)
    replay = N.Replay(base, base, base, base, base, base, None, None)
    grads = base + 65536
    word = {"n1": "n_quantiles", "n65": "n_quantiles", "kappa_neg": "kappa", "kappa_nan": "kappa", "kappa_inf": "kappa",
            "tf32x3": "precision", "dueling": "dueling", "small_scratch": "scratch", "null_scratch": "scratch",
            "misaligned_grads": "grads_out", "null_quantile": "quantile"}[case]
    if case == "n1":
        qr.n_quantiles = 1
    elif case == "n65":
        qr.n_quantiles = 65
    elif case == "kappa_neg":
        qr.kappa = -0.5
    elif case == "kappa_nan":
        qr.kappa = float("nan")
    elif case == "kappa_inf":
        qr.kappa = float("inf")
    elif case == "tf32x3":
        hp.precision = 2
    elif case == "dueling":
        hp.dueling = 1
    elif case == "small_scratch":
        qr.scratch_bytes = sb.value - 1
    elif case == "null_scratch":
        qr.scratch = None
    elif case == "misaligned_grads":
        grads += 4
    qp = None if case == "null_quantile" else C.byref(qr)
    rc = lib.dmdqn_learn_grads_quantile(C.byref(d), C.byref(hp), qp, C.byref(replay), C.byref(nets), base, None, 32, grads,
                                        None, ws_ptr, ws.value, None)
    assert rc == N.ERR_ARG
    assert word in lib.dmdqn_last_error().decode()
    if case in ("n1", "n65", "kappa_neg", "kappa_nan", "kappa_inf", "null_quantile"):
        assert lib.dmdqn_act_quantile(C.byref(d), C.byref(nets), qp, base, 96, base, base, base, base, None, None) == N.ERR_ARG
        assert lib.dmdqn_debug_quantile(C.byref(d), qp, C.byref(N.DistViews())) == N.ERR_ARG
    if case in ("small_scratch", "null_scratch"):
        assert lib.dmdqn_debug_quantile(C.byref(d), C.byref(qr), C.byref(N.DistViews())) == N.ERR_ARG


def test_debug_views_point_into_the_scratch(lib):
    d = N.Dims(2, 2, 89, 96, 64, 4, 32, 100)
    sb = C.c_size_t()
    N.check(lib.dmdqn_dist_scratch_bytes(C.byref(d), 50, C.byref(sb)))
    sc_keep, sc_ptr = _buf(sb.value)
    v = N.DistViews()
    N.check(lib.dmdqn_debug_quantile(C.byref(d), C.byref(N.Quantile(50, 0.0, sc_ptr, sb.value)), C.byref(v)))
    rows = 2 * 32
    up = lambda x: (x + 255) // 256 * 256
    assert v.target_dist == sc_ptr and v.h2 == sc_ptr + up(rows * 52 * 4)
    assert v.dlogits == v.h2 + up(rows * 64 * 4)


# ------------------------------------------------------------------ host configuration ---------------------------------
def _cfg(**kw):
    cfg = dict(DEFAULTS, quantile=True)
    cfg.update(kw)
    return cfg


def test_auto_precision_resolves_to_fp32_and_plain_configs_are_untouched():
    assert quantile_config(_cfg())["precision"] == "fp32"
    assert quantile_config(_cfg(precision="fp32"))["precision"] == "fp32"
    assert quantile_config(_cfg(quantile_kappa=0))["precision"] == "fp32"
    plain = dict(DEFAULTS)
    assert quantile_config(dict(plain)) == plain
    assert dist_config(_cfg()) == _cfg()           # the C51 validator leaves a quantile config alone


@pytest.mark.parametrize("kw,word", [({"precision": "tf32x3"}, "precision"), ({"precision": "tf32"}, "precision"),
                                     ({"distributional": True}, "distributional"), ({"dueling": True}, "dueling"),
                                     ({"noisy": True}, "noisy"), ({"loss": "huber"}, "loss"),
                                     ({"num_quantiles": 1}, "num_quantiles"), ({"num_quantiles": 65}, "num_quantiles"),
                                     ({"num_quantiles": 5.0}, "num_quantiles"), ({"num_quantiles": True}, "num_quantiles"),
                                     ({"quantile_kappa": -1.0}, "quantile_kappa"),
                                     ({"quantile_kappa": float("nan")}, "quantile_kappa"),
                                     ({"quantile_kappa": float("inf")}, "quantile_kappa"),
                                     ({"quantile_kappa": "1"}, "quantile_kappa"), ({"quantile": "yes"}, "quantile")])
def test_host_refusals(kw, word):
    with pytest.raises(ValueError, match=word):
        quantile_config(_cfg(**kw))


def test_defaults_and_config_yaml_have_the_keys():
    import yaml
    assert DEFAULTS["quantile"] is False and DEFAULTS["num_quantiles"] == 50 and DEFAULTS["quantile_kappa"] == 1.0
    path = os.path.join(os.path.dirname(__file__), "..", "config", "agent_config.yaml")
    cfg = yaml.safe_load(open(path))
    assert cfg["quantile"] is False and cfg["num_quantiles"] == 50 and cfg["quantile_kappa"] == 1.0
