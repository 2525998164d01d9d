"""Rainbow networks on the CPU (config ``rainbow``): the oracle against a torch.nn Rainbow module (noisy layers, a dueling
distributional head, softmax over atoms) and float64 autograd, the adjointness of the per-atom fold and projection, the
layout and noise-record offsets, the ABI refusals of every Rainbow call, the config key, the initial weights, and the
shared-parameter Rainbow step over gloo with the oracle standing in for the kernels."""
import ctypes as C
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import noisy_oracle as NO
import rainbow_oracle as RO
from dmdqn_b200.group import DEFAULTS, keras_init, rainbow_config
from dmdqn_b200.parallel import SharedParameterStep


def _rec(dp, h, n):
    npad = (n + 3) // 4 * 4
    off = np.cumsum([0, dp, h, h, h, h, 4 * npad, h, npad])
    return SimpleNamespace(**dict(zip(("w1_in", "w1_out", "w2_in", "w2_out", "w3_in", "w3_out", "v_in", "v_out"), off[:8])),
                           stride=int((off[8] + 31) // 32 * 32))


def _layout(dp, h, n):
    npad = (n + 3) // 4 * 4
    L = SimpleNamespace(w1=0, b1=dp * h)
    L.w2 = L.b1 + h; L.b2 = L.w2 + h * h; L.w3 = L.b2 + h; L.b3 = L.w3 + h * 4 * npad
    L.wv = L.b3 + 4 * npad; L.bv = L.wv + h * npad; L.end = L.bv + npad; L.stride = (L.end + 31) // 32 * 32
    return L


class NoisyLinear(torch.nn.Module):
    """Fortunato et al.'s factorized NoisyLinear (y = x (mu_w + sigma_w * outer(f_in, f_out)) + mu_b + sigma_b * f_out)."""

    def __init__(self, mu_w, mu_b, sig_w, sig_b):
        super().__init__()
        self.mu_w, self.mu_b = torch.nn.Parameter(mu_w.clone()), torch.nn.Parameter(mu_b.clone())
        self.sig_w, self.sig_b = torch.nn.Parameter(sig_w.clone()), torch.nn.Parameter(sig_b.clone())

    def forward(self, x, f_in, f_out):
        return x @ (self.mu_w + self.sig_w * torch.outer(f_in, f_out)) + self.mu_b + self.sig_b * f_out


def _params(seed, d, h, a, n):
    mu = keras_init(seed, d, h, a * n, dueling=True, value_size=n)
    mu[5] = mu[5] + 0.1 * torch.randn(mu[5].shape)
    mu[7] = mu[7] + 0.1 * torch.randn(mu[7].shape)
    sg = [torch.rand_like(p) * 0.1 for p in mu]
    return mu, sg


@pytest.mark.parametrize("a,n", [(4, 11), (3, 51), (2, 2)])
def test_oracle_matches_a_torch_nn_rainbow_module_and_float64_autograd(a, n):
    torch.manual_seed(a + n)
    d, h, b = 89, 64, 16
    rec = _rec(96, h, n)
    record = RO.noise_record(99, 4, 0, rec, d, a, n)
    mu, sg = _params(5, d, h, a, n)
    eps = RO.eps_params(record, rec, d, a, n)
    orc = RO.RainbowOracle(1, d, [h, h], a, n, -10.0, 10.0)
    x = torch.randn(1, b, d) * 0.2
    eff = [p.detach().requires_grad_(True) for p in NO.NoisyStackedOracle.effective([p[None] for p in mu], [p[None] for p in sg],
                                                                                     [e[None] for e in eps])]
    logits = orc.logits(eff, x.numpy())                         # [1, B, A, N]
    f = [torch.as_tensor(v) for v in RO.factors(record, rec)]
    npad = (n + 3) // 4 * 4
    fo = f[5].reshape(4, npad)[:a, :n].reshape(-1)
    layers = [NoisyLinear(mu[2 * i], mu[2 * i + 1], sg[2 * i], sg[2 * i + 1]) for i in range(4)]
    h1 = torch.relu(layers[0](x[0], f[0][:d], f[1]))
    h2 = torch.relu(layers[1](h1, f[2], f[3]))
    adv = layers[2](h2, f[4], fo).reshape(b, a, n)
    val = layers[3](h2, f[6], f[7][:n]).reshape(b, 1, n)
    ref = val + adv - adv.mean(dim=1, keepdim=True)
    torch.testing.assert_close(logits[0], ref, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(torch.softmax(logits[0], -1), torch.softmax(ref, -1), rtol=1e-5, atol=1e-6)
    # gradients of a cross-entropy against fixed targets: the oracle's effective-weight gradient, mapped to mu and sigma by
    # the fold rule, against float64 autograd through the module
    m = torch.softmax(torch.randn(b, a, n), -1)
    g_eff = torch.autograd.grad(-(m * torch.log_softmax(logits[0], -1)).sum(), eff)
    layers64 = [NoisyLinear(*(p.double() for p in (mu[2 * i], mu[2 * i + 1], sg[2 * i], sg[2 * i + 1]))) for i in range(4)]
    f64 = [v.double() for v in f]
    h1 = torch.relu(layers64[0](x[0].double(), f64[0][:d], f64[1]))
    h2 = torch.relu(layers64[1](h1, f64[2], f64[3]))
    adv = layers64[2](h2, f64[4], fo.double()).reshape(b, a, n)
    val = layers64[3](h2, f64[6], f64[7][:n]).reshape(b, 1, n)
    (-(m.double() * torch.log_softmax(val + adv - adv.mean(dim=1, keepdim=True), -1)).sum()).backward()
    for k, l in enumerate(layers64):
        for j, (pm, ps) in enumerate(((l.mu_w, l.sig_w), (l.mu_b, l.sig_b))):
            g = g_eff[2 * k + j][0].double()
            torch.testing.assert_close(g, pm.grad, rtol=1e-4, atol=1e-6)
            torch.testing.assert_close(g * eps[2 * k + j].double(), ps.grad, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("a,n", [(4, 11), (3, 5), (1, 2)])
def test_fold_and_projection_are_adjoint(a, n):
    """<fold(W), G> = <W, project(G)>: the projection is the gradient of the fold."""
    h = 8
    L = _layout(16, h, n)
    rng = np.random.default_rng(a * n)
    blk = np.zeros(L.stride, np.float32)
    npad = (n + 3) // 4 * 4
    blk[L.w3:L.b3].reshape(h, 4, npad)[:, :a, :n] = rng.standard_normal((h, a, n))
    blk[L.b3:L.wv].reshape(4, npad)[:a, :n] = rng.standard_normal((a, n))
    blk[L.wv:L.bv].reshape(h, npad)[:, :n] = rng.standard_normal((h, n))
    blk[L.bv:L.bv + n] = rng.standard_normal(n)
    head = RO.fold_heads(blk, L, h, a, n).astype(np.float64)
    g = np.zeros(L.stride, np.float32)
    g[L.w3:L.wv] = rng.standard_normal(L.wv - L.w3)
    g[L.w3:L.wv].reshape(h + 1, 4, npad)[:, a:] = 0
    g[L.w3:L.wv].reshape(h + 1, 4, npad)[:, :, n:] = 0
    proj = RO.project_heads(g, L, h, a, n).astype(np.float64)
    lhs = float(head @ g[L.w3:L.wv].astype(np.float64))
    rhs = float(blk[L.w3:L.end].astype(np.float64) @ proj[L.w3:L.end])
    assert abs(lhs - rhs) < 1e-4 * max(1.0, abs(lhs))
    assert np.all(proj[L.wv:L.bv].reshape(h, npad)[:, n:] == 0) and np.all(proj[L.bv + n:L.end] == 0)


@pytest.fixture(scope="module")
def lib():
    from dmdqn_b200 import _native as N
    from dmdqn_b200 import build as B
    B.build()
    return N.lib()


@pytest.mark.parametrize("h,n", [(64, 2), (128, 11), (256, 51), (512, 64)])
def test_layout_and_noise_record_offsets(lib, h, n):
    from dmdqn_b200 import _native as N
    d = N.Dims(4, 4, 89, 96, h, 4, 32, 100)
    lay, rec = N.RainbowLayout(), N.NoiseRecord()
    N.check(lib.dmdqn_param_layout_rainbow(C.byref(d), n, C.byref(lay)))
    N.check(lib.dmdqn_noise_layout_rainbow(C.byref(d), n, C.byref(rec)))
    want, wrec = _layout(96, h, n), _rec(96, h, n)
    for k in ("w1", "b1", "w2", "b2", "w3", "b3", "wv", "bv", "end", "stride"):
        assert getattr(lay, k) == getattr(want, k), k
    for k in ("w1_in", "w1_out", "w2_in", "w2_out", "w3_in", "w3_out", "v_in", "v_out", "stride"):
        assert getattr(rec, k) == getattr(wrec, k), k
    c51 = N.Layout()
    N.check(lib.dmdqn_param_layout_dist(C.byref(d), n, C.byref(c51)))
    assert (c51.w3, c51.b3) == (lay.w3, lay.b3) and lay.wv == c51.b3 + 4 * ((n + 3) // 4 * 4)
    sb, sd = C.c_size_t(), C.c_size_t()
    N.check(lib.dmdqn_rainbow_scratch_bytes(C.byref(d), n, C.byref(sb)))
    N.check(lib.dmdqn_dist_scratch_bytes(C.byref(d), n, C.byref(sd)))
    assert sb.value >= sd.value + 2 * 4 * (h + 1) * 4 * ((n + 3) // 4 * 4) * 4


def test_cfg3_numbers(lib):
    from dmdqn_b200 import _native as N
    d = N.Dims(256, 256, 89, 96, 256, 4, 256, 30000)
    lay = N.RainbowLayout()
    N.check(lib.dmdqn_param_layout_rainbow(C.byref(d), 51, C.byref(lay)))
    assert (lay.wv, lay.end, lay.stride) == (144080, 157444, 157472)


def _buf(n=1 << 16):
    raw = (C.c_char * (n + 256))()
    return raw, (C.addressof(raw) + 255) // 256 * 256


@pytest.mark.parametrize("case", ["atoms1", "atoms65", "vmin_ge_vmax", "nan", "tf32x3", "dueling0", "small_scratch",
                                  "null_sigma_m", "misaligned_grads"])
def test_abi_refusals(lib, case):
    from dmdqn_b200 import _native as N
    d = N.Dims(2, 2, 89, 96, 64, 4, 32, 100)
    keep, base = _buf(1 << 22)
    ws = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(d), C.byref(ws)))
    ws_keep, ws_ptr = _buf(ws.value)
    sb = C.c_size_t()
    N.check(lib.dmdqn_rainbow_scratch_bytes(C.byref(d), 11, C.byref(sb)))
    sc_keep, sc_ptr = _buf(sb.value)
    dist_ = N.Dist(11, -10.0, 10.0, sc_ptr, sb.value)
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 10, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100, 1, dueling=1)
    nets = N.Nets(base, base + 4096, base + 8192, base + 12288, base + 16384)
    noisy = N.Noisy(*(base + 20480 + 4096 * k for k in range(8)))
    replay = N.Replay(base, base, base, base, base, base, None, None)
    grads = base + 65536
    if case == "atoms1":
        dist_.n_atoms = 1
    elif case == "atoms65":
        dist_.n_atoms = 65
    elif case == "vmin_ge_vmax":
        dist_.v_min = 10.0
    elif case == "nan":
        dist_.v_max = float("nan")
    elif case == "tf32x3":
        hp.precision = 2
    elif case == "dueling0":
        hp.dueling = 0
    elif case == "small_scratch":
        dist_.scratch_bytes = sb.value - 1
    elif case == "null_sigma_m":
        noisy.sigma_m = None
    elif case == "misaligned_grads":
        grads += 4
    n_atoms = dist_.n_atoms
    rc = lib.dmdqn_learn_grads_rainbow(C.byref(d), C.byref(hp), C.byref(dist_), C.byref(replay), C.byref(nets), C.byref(noisy),
                                       base, None, 32, grads, None, ws_ptr, ws.value, None)
    assert rc == N.ERR_ARG, lib.dmdqn_last_error()
    if case in ("atoms1", "atoms65", "tf32x3", "dueling0", "null_sigma_m", "misaligned_grads"):
        assert lib.dmdqn_adam_apply_rainbow(C.byref(d), C.byref(hp), C.byref(nets), C.byref(noisy), n_atoms, grads, ws_ptr,
                                            ws.value, None) == N.ERR_ARG
    if case in ("atoms1", "atoms65"):
        for fn, out in ((lib.dmdqn_param_layout_rainbow, N.RainbowLayout()), (lib.dmdqn_noise_layout_rainbow, N.NoiseRecord())):
            assert fn(C.byref(d), n_atoms, C.byref(out)) == N.ERR_ARG
        assert lib.dmdqn_rainbow_scratch_bytes(C.byref(d), n_atoms, C.byref(C.c_size_t())) == N.ERR_ARG
        assert lib.dmdqn_sync_target_rainbow(C.byref(d), C.byref(nets), C.byref(noisy), n_atoms, None, -1.0, None) == N.ERR_ARG
    if case in ("atoms1", "atoms65", "vmin_ge_vmax", "nan", "small_scratch"):
        assert lib.dmdqn_rainbow_fold(C.byref(d), C.byref(dist_), C.byref(nets), C.byref(noisy), None) == N.ERR_ARG
        assert lib.dmdqn_debug_rainbow(C.byref(d), C.byref(dist_), C.byref(N.RainbowViews())) == N.ERR_ARG
    if case in ("atoms1", "atoms65", "vmin_ge_vmax", "nan"):
        assert lib.dmdqn_act_rainbow(C.byref(d), C.byref(nets), C.byref(noisy), C.byref(dist_), base, 96, base, base, base, base,
                                     None, None) == N.ERR_ARG
    if case == "null_sigma_m":
        noisy.sigma = None
        assert lib.dmdqn_sync_target_rainbow(C.byref(d), C.byref(nets), C.byref(noisy), 11, None, -1.0, None) == N.ERR_ARG
        assert lib.dmdqn_rainbow_fold(C.byref(d), C.byref(dist_), C.byref(nets), C.byref(noisy), None) == N.ERR_ARG
        assert lib.dmdqn_act_rainbow(C.byref(d), C.byref(nets), C.byref(noisy), C.byref(dist_), base, 96, base, base, base, base,
                                     None, None) == N.ERR_ARG


def _cfg(**kw):
    cfg = dict(DEFAULTS, rainbow=True)
    cfg.update(kw)
    return cfg


def test_config_default_yaml_and_precision():
    import yaml
    assert DEFAULTS["rainbow"] is False
    path = os.path.join(os.path.dirname(__file__), "..", "config", "agent_config.yaml")
    assert yaml.safe_load(open(path))["rainbow"] is False
    assert rainbow_config(_cfg())["precision"] == "fp32"
    assert rainbow_config(_cfg(precision="fp32"))["precision"] == "fp32"
    plain = dict(DEFAULTS)
    assert rainbow_config(dict(plain)) == plain


@pytest.mark.parametrize("kw,word", [({"distributional": True}, "distributional"), ({"quantile": True}, "quantile"),
                                     ({"iqn": True}, "iqn"), ({"dueling": True}, "dueling"), ({"noisy": True}, "noisy"),
                                     ({"precision": "tf32x3"}, "precision"), ({"precision": "tf32"}, "precision"),
                                     ({"loss": "huber"}, "loss"), ({"global_clipnorm": 1.0}, "global_clipnorm"),
                                     ({"num_atoms": 1}, "num_atoms"), ({"num_atoms": 65}, "num_atoms"),
                                     ({"v_min": 1.0, "v_max": 1.0}, "v_min"), ({"rainbow": "yes"}, "rainbow")])
def test_config_refusals(kw, word):
    with pytest.raises(ValueError, match=word):
        rainbow_config(_cfg(**kw))


def test_w1_to_b3_are_drawn_as_a_c51_groups_and_wv_after_them():
    for seed in (0, 7):
        rb = keras_init(seed, 89, 64, 4 * 51, dueling=True, value_size=51)
        c51 = keras_init(seed, 89, 64, 4 * 51)
        assert len(rb) == 8 and all(torch.equal(x, y) for x, y in zip(rb[:6], c51))
        assert tuple(rb[6].shape) == (64, 51) and torch.all(rb[7] == 0)
        assert rb[6].abs().max() <= (6.0 / (64 + 51)) ** 0.5


# ------------------------------------------------------------------ gloo, world size 2 ----------------------------------
H, A, NA, B_GLOBAL, KEY = 64, 4, 11, 32, 0x0123_4567_89ab_cdef


def _data():
    rng = np.random.default_rng(0)
    S = (rng.standard_normal((1, B_GLOBAL, 89)) * 0.3).astype(np.float32)
    S2 = (rng.standard_normal((1, B_GLOBAL, 89)) * 0.3).astype(np.float32)
    A_ = rng.integers(0, A, (1, B_GLOBAL)); R = rng.standard_normal((1, B_GLOBAL)).astype(np.float32)
    D = (rng.random((1, B_GLOBAL)) < 0.1).astype(np.float32)
    return S, A_, R, S2, D


def _eps(t, s):
    rec = _rec(96, H, NA)
    return [e[None] for e in RO.eps_params(RO.noise_record(KEY, t, s, rec, 89, A, NA), rec, 89, A, NA)]


def _oracle():
    orc = RO.RainbowOracle(1, 89, [H, H], A, NA, -10.0, 10.0, seed0=3)
    mu = [p[None] for p in keras_init(3, 89, H, A * NA, dueling=True, value_size=NA)]
    sg = [torch.full_like(p, 0.05) for p in mu]
    orc.set_state(mu, sg, [p.clone() for p in mu], [p.clone() for p in sg], *([torch.zeros_like(p) for p in mu] for _ in range(4)))
    return orc


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from oracle.dqn import adam_scalars, adam_update_
        torch.set_num_threads(1)
        b_local = B_GLOBAL // world
        S, A_, R, S2, D = _data()
        sl = slice(rank * b_local, (rank + 1) * b_local)
        orc = _oracle()

        def local_grads(global_batch):     # dmdqn_learn_grads_rainbow: the gradient of the effective weights
            t = int(orc.learn_step[0])
            out = orc.learn_on_batch(S[:, sl], A_[:, sl], R[:, sl], S2[:, sl], D[:, sl], _eps(t, 0), _eps(t, 1),
                                     loss_batch=global_batch, apply=False)
            metrics = torch.zeros(1, 8); metrics[0, 0] = float(out["loss"][0])
            return torch.cat([torch.as_tensor(g).reshape(-1) for g in out["g_mu"]]), metrics

        def apply(flat):                  # dmdqn_adam_apply_rainbow on the all-reduced block
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


def test_shared_parameter_rainbow_step_equals_single_process_big_batch_step():
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
    for w0, w1 in zip(results[0][1], results[1][1]):
        assert np.array_equal(w0, w1)
