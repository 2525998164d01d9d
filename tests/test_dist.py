"""CPU checks of distributional Q-learning (C51): the oracle's projection and gradients, the host-side configuration and
the C ABI's layout, scratch query and refusals (no GPU needed: every refusal happens before a launch)."""
import ctypes as C

import numpy as np
import pytest
import torch

import dist_oracle as DO
from dmdqn_b200 import _native as N
from dmdqn_b200 import build as B
from dmdqn_b200.group import DEFAULTS, dist_config


@pytest.fixture(scope="module")
def lib():
    B.build()
    return N.lib()


def _p(rng, n):
    x = rng.standard_normal(n).astype(np.float32)
    return DO.probs(x)


# ------------------------------------------------------------------ projection -----------------------------------------
@pytest.mark.parametrize("n", [2, 11, 51])
def test_projection_known_cases(n):
    rng = np.random.default_rng(n)
    z, lo, hi, dz = DO.support(n, -10.0, 10.0)
    p = _p(rng, n)
    r = np.float32(3.3)                       # d = 0: all mass on floor / ceil of b(R)
    m = DO.project(p, r, 0.0, z, lo, hi, dz)
    b = min(np.float32(np.float32(r - lo) / dz), np.float32(n - 1))
    l, u = int(np.floor(b)), int(np.ceil(b))
    assert set(np.nonzero(m)[0]) <= {l, u} and abs(m.sum() - 1) < 1e-6
    assert DO.project(p, 25.0, 0.5, z, lo, hi, dz)[-1] == pytest.approx(1, abs=1e-6)   # above v_max: the last atom
    assert DO.project(p, -25.0, 0.5, z, lo, hi, dz)[0] == pytest.approx(1, abs=1e-6)   # below v_min: the first atom
    k = n // 2                                # R on an atom, d = 0: all mass on that atom
    m = DO.project(p, z[k], 0.0, z, lo, hi, dz)
    assert m[k] == pytest.approx(1, abs=1e-6) and np.abs(np.delete(m, k)).max() < 1e-6


@pytest.mark.parametrize("n", [2, 11, 51, 64])
def test_projection_conserves_mass_and_matches_algorithm_1(n):
    rng = np.random.default_rng(100 + n)
    z, lo, hi, dz = DO.support(n, -7.5, 12.0)
    for _ in range(50):
        p = _p(rng, n)
        r, d = np.float32(rng.uniform(-20, 20)), np.float32(rng.choice([0.0, 0.99, 0.970299, rng.uniform(0, 1)]))
        m = DO.project(p, r, d, z, lo, hi, dz)
        assert abs(float(m.sum(dtype=np.float64)) - 1.0) < 1e-6
        ref = DO.project_float64(p.astype(np.float64), float(r), float(d), z.astype(np.float64), -7.5, 12.0)
        assert np.abs(m - ref).max() < 1e-5


# ------------------------------------------------------------------ gradients ------------------------------------------
def test_oracle_gradients_match_autograd_of_the_cross_entropy():
    """The oracle's logit gradient and its W / b gradients against float64 autograd of mean_i w_i CE_i."""
    rng = np.random.default_rng(7)
    n_atoms, a, b, d, h = 11, 3, 16, 89, 64
    o = DO.DistOracle(2, d, [h, h], a, n_atoms, -5.0, 5.0, seed0=3)
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
    m = torch.as_tensor(out["m"], dtype=torch.float64)
    params = [p.detach().double().requires_grad_(True) for p in o.online]
    x = o.forward(params, torch.as_tensor(s, dtype=torch.float64)).reshape(2, b, a, n_atoms)
    xa = torch.gather(x, 2, torch.as_tensor(act)[..., None, None].expand(2, b, 1, n_atoms))[:, :, 0]
    ce = -(m * torch.log_softmax(xa, dim=-1)).sum(-1)
    loss = (torch.as_tensor(w, dtype=torch.float64) * ce).mean(1).sum()
    gx = torch.autograd.grad(loss, [x], retain_graph=True)[0]
    assert np.abs(out["dlogits"] - gx.reshape(2, b, a, n_atoms).numpy()).max() < 1e-6
    grads = torch.autograd.grad(loss, params)
    for k, (g, ref) in enumerate(zip(out["grads"], grads)):
        assert np.abs(g - ref.numpy()).max() <= 1e-6 * max(1.0, float(ref.abs().max())), k
    ref_ce = ce.detach().numpy()
    assert np.abs(out["ce"] - ref_ce).max() < 1e-6 * np.abs(ref_ce).max()


class TorchC51:
    """An independent float64 C51 learner (torch.nn, textbook softmax / projection / cross-entropy) for comparison."""

    def __init__(self, params, target, n_atoms, v_min, v_max, a, gamma=0.99, lr=5e-4):
        self.p = [t.detach().double().clone().requires_grad_(True) for t in params]
        self.t = [t.detach().double().clone() for t in target]
        self.n, self.a, self.v_min, self.v_max, self.gamma = n_atoms, a, v_min, v_max, gamma
        self.z = torch.linspace(v_min, v_max, n_atoms, dtype=torch.float64)
        self.opt = torch.optim.Adam(self.p, lr=lr, betas=(0.9, 0.999), eps=1e-8)

    def net(self, params, x):
        h = torch.relu(x @ params[0] + params[1])
        h = torch.relu(h @ params[2] + params[3])
        return (h @ params[4] + params[5]).reshape(*x.shape[:-1], self.a, self.n)

    def step(self, s, act, r, s2, disc):
        with torch.no_grad():
            po = torch.softmax(self.net(self.p, s2), -1)
            pt = torch.softmax(self.net(self.t, s2), -1)
            best = (po * self.z).sum(-1).argmax(-1)
            p = pt[torch.arange(s.shape[0]), best]
            tz = (r[:, None] + disc[:, None] * self.z).clamp(self.v_min, self.v_max)
            b = (tz - self.v_min) / ((self.v_max - self.v_min) / (self.n - 1))
            l, u = b.floor().long(), b.ceil().long()
            m = torch.zeros_like(p)
            eq = (l == u).double()
            m.scatter_add_(1, l, p * (u.double() - b + eq))
            m.scatter_add_(1, u, p * (b - l.double()))
        x = self.net(self.p, s)[torch.arange(s.shape[0]), act]
        loss = -(m * torch.log_softmax(x, -1)).sum(-1).mean()
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        return float(loss.detach())


def test_a_few_oracle_steps_match_an_independent_float64_learner():
    rng = np.random.default_rng(11)
    n_atoms, a, b, d, h = 11, 4, 32, 89, 64
    o = DO.DistOracle(1, d, [h, h], a, n_atoms, -10.0, 10.0, seed0=5, target_update_frequency=1000, adam_form="torch")
    ref = TorchC51([p[0] for p in o.online], [p[0] for p in o.target], n_atoms, -10.0, 10.0, a)
    for step in range(3):
        s = rng.integers(-1, 20, (1, b, d)).astype(np.float32)
        s2 = rng.integers(-1, 20, (1, b, d)).astype(np.float32)
        act = rng.integers(0, a, (1, b))
        r = rng.uniform(-3, 3, (1, b)).astype(np.float32)
        disc = np.full((1, b), 0.99, np.float32)
        out = o.learn_on_batch(s, act, r, s2, None, discounts=disc)
        lr = ref.step(torch.as_tensor(s[0], dtype=torch.float64), torch.as_tensor(act[0]), torch.as_tensor(r[0], dtype=torch.float64),
                      torch.as_tensor(s2[0], dtype=torch.float64), torch.as_tensor(disc[0], dtype=torch.float64))
        assert abs(out["loss"][0] - lr) < 1e-5 * max(1.0, abs(lr)), step
        for k, (p, q) in enumerate(zip(o.online, ref.p)):
            assert np.abs(p[0].numpy() - q.detach().numpy()).max() < 1e-5, (step, k)


# ------------------------------------------------------------------ C ABI (no GPU) -------------------------------------
DIMS = (8, 8, 89, 96, 256, 4, 128, 1000)


def test_layout_offsets(lib):
    d = N.Dims(*DIMS)
    lay = N.Layout()
    N.check(lib.dmdqn_param_layout_dist(C.byref(d), 51, C.byref(lay)))
    w3 = 96 * 256 + 256 + 256 * 256 + 256
    assert (lay.w1, lay.b1, lay.w2, lay.b2, lay.w3) == (0, 96 * 256, 96 * 256 + 256, 96 * 256 + 256 + 65536, w3)
    assert lay.b3 == w3 + 256 * 208 and lay.stride == 144096
    plain = N.Layout()
    N.check(lib.dmdqn_param_layout(C.byref(d), C.byref(plain)))
    assert plain.stride == 91680
    for n, np_ in ((2, 4), (11, 12), (64, 64)):
        N.check(lib.dmdqn_param_layout_dist(C.byref(d), n, C.byref(lay)))
        assert lay.b3 == w3 + 256 * 4 * np_ and lay.stride % 32 == 0 and lay.stride >= lay.b3 + 4 * np_


def test_scratch_size(lib):
    d = N.Dims(*DIMS)
    nb = C.c_size_t()
    N.check(lib.dmdqn_dist_scratch_bytes(C.byref(d), 51, C.byref(nb)))
    rows = 8 * 128
    up = lambda x: (x + 255) // 256 * 256
    assert nb.value == up(rows * 52 * 4) + up(rows * 256 * 4) + up(rows * 208 * 4)
    assert lib.dmdqn_dist_scratch_bytes(C.byref(d), 65, C.byref(nb)) == N.ERR_ARG


def _buf(n=1 << 16):
    raw = (C.c_char * (n + 256))()
    return raw, (C.addressof(raw) + 255) // 256 * 256


@pytest.mark.parametrize("case", ["atoms1", "atoms65", "vmin_ge_vmax", "nan", "tf32x3", "dueling", "small_scratch",
                                  "misaligned_grads"])
def test_abi_refusals(lib, case):
    d = N.Dims(2, 2, 89, 96, 64, 4, 32, 100)
    keep, base = _buf(1 << 22)
    ws = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(d), C.byref(ws)))
    ws_keep, ws_ptr = _buf(ws.value)
    sb = C.c_size_t()
    N.check(lib.dmdqn_dist_scratch_bytes(C.byref(d), 11, C.byref(sb)))
    sc_keep, sc_ptr = _buf(sb.value)
    dist = N.Dist(11, -10.0, 10.0, sc_ptr, sb.value)
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 10, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100, 1)
    nets = N.Nets(base, base + 4096, base + 8192, base + 12288, base + 16384)
    replay = N.Replay(base, base, base, base, base, base, None, None)
    grads = base + 65536
    if case == "atoms1":
        dist.n_atoms = 1
    elif case == "atoms65":
        dist.n_atoms = 65
    elif case == "vmin_ge_vmax":
        dist.v_min = 10.0
    elif case == "nan":
        dist.v_max = float("nan")
    elif case == "tf32x3":
        hp.precision = 2
    elif case == "dueling":
        hp.dueling = 1
    elif case == "small_scratch":
        dist.scratch_bytes = sb.value - 1
    elif case == "misaligned_grads":
        grads += 4
    rc = lib.dmdqn_learn_grads_dist(C.byref(d), C.byref(hp), C.byref(dist), C.byref(replay), C.byref(nets), base, None, 32,
                                    grads, None, ws_ptr, ws.value, None)
    assert rc == N.ERR_ARG, lib.dmdqn_last_error()
    if case in ("atoms1", "atoms65"):
        assert lib.dmdqn_param_layout_dist(C.byref(d), dist.n_atoms, C.byref(N.Layout())) == N.ERR_ARG
        assert lib.dmdqn_sync_target_dist(C.byref(d), C.byref(nets), dist.n_atoms, None, -1.0, None) == N.ERR_ARG
        assert lib.dmdqn_adam_apply_dist(C.byref(d), C.byref(hp), C.byref(nets), dist.n_atoms, grads, 0.0, None, ws_ptr,
                                         ws.value, None) == N.ERR_ARG
    if case in ("atoms1", "atoms65", "vmin_ge_vmax", "nan"):
        assert lib.dmdqn_act_dist(C.byref(d), C.byref(nets), C.byref(dist), base, 96, base, base, base, base, None,
                                  None) == N.ERR_ARG
    if case in ("tf32x3", "dueling", "misaligned_grads"):
        assert lib.dmdqn_adam_apply_dist(C.byref(d), C.byref(hp), C.byref(nets), 11, grads, 0.0, None, ws_ptr, ws.value,
                                         None) == N.ERR_ARG


@pytest.mark.parametrize("clip", [-1.0, float("nan"), float("inf")])
def test_adam_apply_dist_refuses_a_bad_clipnorm(lib, clip):
    d = N.Dims(2, 2, 89, 96, 64, 4, 32, 100)
    keep, base = _buf(1 << 20)
    ws = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(d), C.byref(ws)))
    ws_keep, ws_ptr = _buf(ws.value)
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 10, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100, 1)
    nets = N.Nets(base, base + 4096, base + 8192, base + 12288, base + 16384)
    assert lib.dmdqn_adam_apply_dist(C.byref(d), C.byref(hp), C.byref(nets), 11, base + 65536, clip, None, ws_ptr, ws.value,
                                     None) == N.ERR_ARG
    assert "global_clipnorm" in lib.dmdqn_last_error().decode()


# ------------------------------------------------------------------ host configuration ---------------------------------
def _cfg(**kw):
    cfg = dict(DEFAULTS, distributional=True)
    cfg.update(kw)
    return cfg


def test_auto_precision_resolves_to_fp32_and_plain_configs_are_untouched():
    assert dist_config(_cfg())["precision"] == "fp32"
    assert dist_config(_cfg(precision="fp32"))["precision"] == "fp32"
    plain = dict(DEFAULTS)
    assert dist_config(dict(plain)) == plain


@pytest.mark.parametrize("kw,word", [({"precision": "tf32x3"}, "precision"), ({"precision": "tf32"}, "precision"),
                                     ({"dueling": True}, "dueling"), ({"noisy": True}, "noisy"), ({"loss": "huber"}, "loss"),
                                     ({"num_atoms": 1}, "num_atoms"), ({"num_atoms": 65}, "num_atoms"),
                                     ({"num_atoms": 5.5}, "num_atoms"), ({"v_min": 1.0, "v_max": 1.0}, "v_min"),
                                     ({"v_max": float("inf")}, "v_max"), ({"distributional": "yes"}, "distributional")])
def test_host_refusals(kw, word):
    with pytest.raises(ValueError, match=word):
        dist_config(_cfg(**kw))


def test_config_yaml_has_the_keys():
    import yaml
    import os
    path = os.path.join(os.path.dirname(__file__), "..", "config", "agent_config.yaml")
    cfg = yaml.safe_load(open(path))
    assert cfg["distributional"] is False and cfg["num_atoms"] == 51 and cfg["v_min"] == -10.0 and cfg["v_max"] == 10.0
