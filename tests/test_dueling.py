"""Dueling Q-networks (config ``dueling``) on the CPU: the oracle against an independent torch.nn two-stream module, the
fold identity and the gradient projection the kernels use, the parameter layout and the hparams field of the C ABI, the
refusals, and the config / init plumbing."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from dueling_oracle import DuelingStackedOracle, dueling_init, fold_np, project_np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


class TwoStream(torch.nn.Module):
    """The dueling architecture as torch.nn layers: shared Dense(relu) x 2, then value and advantage streams."""

    def __init__(self, d, h, a):
        super().__init__()
        self.l1, self.l2 = torch.nn.Linear(d, h), torch.nn.Linear(h, h)
        self.adv, self.val = torch.nn.Linear(h, a), torch.nn.Linear(h, 1)

    def forward(self, x):
        h = torch.relu(self.l2(torch.relu(self.l1(x))))
        adv = self.adv(h)
        return self.val(h) + (adv - adv.mean(dim=-1, keepdim=True))

    def load(self, p):
        with torch.no_grad():
            for lin, w, b in ((self.l1, p[0], p[1]), (self.l2, p[2], p[3]), (self.adv, p[4], p[5]), (self.val, p[6], p[7])):
                lin.weight.copy_(w.T)
                lin.bias.copy_(b)


def _random_params(seed, d, h, a, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    shapes = [(d, h), (h,), (h, h), (h,), (h, a), (a,), (h, 1), (1,)]
    return [torch.randn(s, generator=g, dtype=dtype) * 0.3 for s in shapes]


@pytest.mark.parametrize("a", [1, 2, 3, 4])
def test_oracle_forward_and_gradients_match_a_torch_nn_two_stream_module(a):
    d, h, b = 7, 16, 9
    orc = DuelingStackedOracle(1, d, [h, h], a, seed0=3)
    p = [t[0].clone() for t in orc.online]
    net = TwoStream(d, h, a)
    net.load(p)
    x = torch.randn(1, b, d, generator=torch.Generator().manual_seed(1))
    q = orc.forward([t.clone() for t in orc.online], x)
    assert torch.allclose(q[0], net(x[0]), rtol=1e-5, atol=1e-6)
    params = [t.detach().clone().requires_grad_(True) for t in orc.online]
    orc.forward(params, x)[0, :, a - 1].square().sum().backward()
    net(x[0])[:, a - 1].square().sum().backward()
    mods = (net.l1, net.l2, net.adv, net.val)
    for k, mod in enumerate(mods):
        assert torch.allclose(params[2 * k].grad[0], mod.weight.grad.T, rtol=1e-4, atol=1e-6), k
        assert torch.allclose(params[2 * k + 1].grad[0], mod.bias.grad, rtol=1e-4, atol=1e-6), k


def _folded(p, a):
    """W3e [H, 4], b3e [4] in float64 from the textbook parameters (the header's formula)."""
    w3 = torch.zeros(p[4].shape[0], 4, dtype=p[4].dtype)
    w3[:, :a] = p[4] - p[4].mean(dim=1, keepdim=True) + p[6]
    b3 = torch.zeros(4, dtype=p[4].dtype)
    b3[:a] = p[5] - p[5].mean() + p[7]
    return w3, b3


@pytest.mark.parametrize("a", [1, 2, 3, 4])
def test_fold_identity_holds_in_float64_and_within_rounding_in_fp32(a):
    d, h = 5, 32
    p = _random_params(a, d, h, a)
    x = torch.randn(1, 40, d, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    q = DuelingStackedOracle.forward([t[None] for t in p], x)[0]
    h2 = torch.relu(torch.relu(x[0] @ p[0] + p[1]) @ p[2] + p[3])
    w3e, b3e = _folded(p, a)
    assert torch.allclose(h2 @ w3e[:, :a] + b3e[:a], q, rtol=1e-12, atol=1e-12)
    assert torch.all(w3e[:, a:] == 0) and torch.all(b3e[a:] == 0)
    f = [t.float().numpy() for t in p]
    w3 = np.zeros((h, 4), np.float32); w3[:, :a] = f[4]
    b3 = np.zeros(4, np.float32); b3[:a] = f[5]
    w3e32, b3e32 = fold_np(w3, b3, f[6][:, 0], f[7][0], a)
    q32 = h2.float().numpy() @ w3e32[:, :a] + b3e32[:a]
    assert np.allclose(q32, q.numpy(), rtol=1e-5, atol=1e-5)
    assert np.all(w3e32[:, a:] == 0) and np.all(b3e32[a:] == 0)


@pytest.mark.parametrize("a", [1, 2, 3, 4])
def test_projection_of_the_folded_gradient_equals_autograd(a):
    d, h = 5, 24
    p = [t.requires_grad_(True) for t in _random_params(10 + a, d, h, a)]
    x = torch.randn(1, 30, d, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    act = torch.randint(0, a, (30,), generator=torch.Generator().manual_seed(4))
    q = DuelingStackedOracle.forward([t[None] for t in p], x)[0]
    loss = (q.gather(1, act[:, None])[:, 0] - 0.5).square().mean()
    grads = torch.autograd.grad(loss, p)
    # G = dL/dW3e, dL/db3e of the equivalent plain head (columns >= A never taken: exactly zero)
    w3e, b3e = [t.detach().requires_grad_(True) for t in _folded([t.detach() for t in p], a)]
    h2 = torch.relu(torch.relu(x[0] @ p[0].detach() + p[1].detach()) @ p[2].detach() + p[3].detach())
    qe = h2 @ w3e + b3e
    lossp = (qe.gather(1, act[:, None])[:, 0] - 0.5).square().mean()
    g3, gb = torch.autograd.grad(lossp, [w3e, b3e])
    assert torch.all(g3[:, a:] == 0) and torch.all(gb[a:] == 0)
    dw3 = g3 - g3[:, :a].sum(dim=1, keepdim=True) / a
    db3 = gb - gb[:a].sum() / a
    assert torch.allclose(dw3[:, :a], grads[4], rtol=1e-10, atol=1e-12)
    assert torch.allclose(db3[:a], grads[5], rtol=1e-10, atol=1e-12)
    assert torch.allclose(g3[:, :a].sum(dim=1), grads[6][:, 0], rtol=1e-10, atol=1e-12)
    assert torch.allclose(gb[:a].sum(), grads[7][0], rtol=1e-10, atol=1e-12)
    # the fp32 restatement the GPU tests use agrees and keeps the advantage columns >= A at exactly zero
    pw3, pb3, pwv, pbv = project_np(g3.float().numpy(), gb.float().numpy(), a)
    assert np.all(pw3[:, a:] == 0) and np.all(pb3[a:] == 0)
    assert np.allclose(pw3[:, :a], grads[4].numpy(), rtol=1e-5, atol=1e-7)
    assert np.allclose(pwv, grads[6][:, 0].numpy(), rtol=1e-5, atol=1e-7)
    assert np.allclose(pbv, grads[7][0].item(), rtol=1e-5, atol=1e-7)


@pytest.fixture(scope="module")
def lib():
    from dmdqn_b200 import _native as N
    from dmdqn_b200 import build as B
    B.build()
    return N.lib()


@pytest.mark.parametrize("h,stride", [(64, 96), (128, 96), (256, 96), (512, 96), (256, 32), (64, 128)])
def test_dueling_layout_keeps_the_plain_offsets_and_adds_the_value_head(lib, h, stride):
    from dmdqn_b200 import _native as N
    d = N.Dims(8, 8, min(89, stride), stride, h, 4, 64, 100)
    plain, duel = N.Layout(), N.DuelingLayout()
    N.check(lib.dmdqn_param_layout(C.byref(d), C.byref(plain)))
    N.check(lib.dmdqn_param_layout_dueling(C.byref(d), C.byref(duel)))
    for k in ("w1", "b1", "w2", "b2", "w3", "b3"):
        assert getattr(plain, k) == getattr(duel, k), k
    assert plain.b3 == stride * h + h + h * h + h + 4 * h
    assert plain.stride == (plain.b3 + 4 + 31) // 32 * 32            # the plain layout is unchanged
    assert duel.wv == duel.b3 + 4 and duel.wv % 4 == 0 and duel.bv == duel.b3 + 4 + h
    assert duel.stride % 32 == 0 and duel.stride >= duel.b3 + 8 + h and duel.stride - (duel.b3 + 8 + h) < 32


def test_hparams_keeps_its_size_with_dueling_in_the_interior_padding():
    from dmdqn_b200 import _native as N
    assert C.sizeof(N.HParams) == 112 and N.HParams.dueling.offset == 76
    assert N.HParams.precision.offset == 72 and N.HParams.per_alpha.offset == 80 and N.HParams.n_step.offset == 108
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 1000, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100)
    assert (hp.per_alpha, hp.per_beta_steps, hp.n_step, hp.dueling) == (0.6, 100, 0, 0)
    assert N.HParams(0.99, dueling=1).dueling == 1
    with pytest.raises(TypeError, match="keyword-only"):
        N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 1000, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100, 1, 1)


def test_native_calls_refuse_a_bad_dueling_flag_before_launching_anything(lib):
    from dmdqn_b200 import _native as N
    dims = N.Dims(4, 4, 89, 96, 64, 4, 32, 100)
    nbytes = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(dims), C.byref(nbytes)))
    ws = (C.c_uint8 * 256)()           # never touched: validation fails before anything is launched
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 1000, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100, 1, dueling=2)
    replay, nets = N.Replay(1, 1, 1, 1, 1, 1, None, None), N.Nets(1, 1, 1, 1, 1)
    w, nb = C.addressof(ws), nbytes.value
    peers = N.Peers()
    peers.world, peers.epoch = 1, 1
    for p in range(1):
        peers.grads[p], peers.loss[p], peers.flags[p] = w, w, w
    one = N.Dims(1, 1, 89, 96, 64, 4, 32, 100)
    N.check(lib.dmdqn_workspace_bytes(C.byref(one), C.byref(nbytes)))
    calls = {
        "learn": lambda: lib.dmdqn_learn(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets), w, None, None, w, nb, None),
        "learn_stages": lambda: lib.dmdqn_learn_stages(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets), w, None,
                                                       None, w, nb, 15, None),
        "sample": lambda: lib.dmdqn_sample(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets), w, None, 0, w, nb, None),
        "learn_grads": lambda: lib.dmdqn_learn_grads(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets), w, None, 32,
                                                     w, w, w, nb, None),
        "step_host": lambda: lib.dmdqn_step_host(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets),
                                                 C.byref(N.StepBlock(256, 0, 16, 32, 48, 64, 80, 89)), w, w, w, w, w, nb, None),
        "adam_apply": lambda: lib.dmdqn_adam_apply(C.byref(dims), C.byref(hp), C.byref(nets), w, w, nb, None),
        "clip_adam_apply": lambda: lib.dmdqn_clip_adam_apply(C.byref(dims), C.byref(hp), C.byref(nets), w, 1.0, None, w, nb,
                                                             None),
        "allreduce_adam": lambda: lib.dmdqn_allreduce_adam(C.byref(one), C.byref(hp), C.byref(nets), C.byref(peers), w, None,
                                                           w, nbytes.value, None),
    }
    for name, call in calls.items():
        assert call() == N.ERR_ARG, name
        assert "dueling=2" in lib.dmdqn_last_error().decode(), name


def test_config_key_defaults_off_and_bad_values_are_refused():
    import yaml
    from dmdqn_b200.group import DEFAULTS, AgentGroup
    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "agent_config.yaml")))
    assert cfg["dueling"] is False and DEFAULTS["dueling"] is False
    for bad in (2, "yes", None):
        with pytest.raises(ValueError, match="dueling"):
            AgentGroup(2, {"nn_layers": [64, 64], "dueling": bad})


@pytest.mark.parametrize("a", [2, 4])
def test_keras_init_draws_the_plain_weights_first_and_the_value_head_after_them(a):
    from dmdqn_b200.group import keras_init
    plain = keras_init(7, 89, 64, a)
    duel = keras_init(7, 89, 64, a, dueling=True)
    assert len(plain) == 6 and len(duel) == 8
    for p, q in zip(plain, duel):
        assert torch.equal(p, q)
    assert duel[6].shape == (64, 1) and duel[7].shape == (1,) and torch.all(duel[7] == 0)
    limit = np.sqrt(6.0 / 65)
    assert float(duel[6].abs().max()) <= limit and float(duel[6].std()) > 0
    assert all(torch.equal(x, y) for x, y in zip(duel, dueling_init(7, 89, 64, a)))
