"""CPU: the hidden-width envelope of DQN (every multiple of 128 up to 1024), its arenas at each width, and the oracle
against the reference fixture recorded at hidden 256 (tests/golden/iqn_hidden256.npz, tools/make_golden_hidden.py)."""
import os

import numpy as np
import pytest
import torch

from helpers import make_args
from oracle import cases, losses, network as net

WIDTHS = (128, 256, 384, 512, 640, 768, 896, 1024)


def _dqn(hidden, rainbow_only=False, action_space=18):
    from rainbow_iqn_apex_b200.model import DQN
    args = make_args(torch.device("cpu"), rainbow_only=rainbow_only)
    args.hidden_size = hidden
    return DQN(args, action_space)


def test_envelope_constant():
    from rainbow_iqn_apex_b200 import model
    assert model.HIDDEN_SIZES == WIDTHS


@pytest.mark.parametrize("rainbow_only", [False, True])
@pytest.mark.parametrize("hidden", WIDTHS)
def test_state_dict_and_arenas(hidden, rainbow_only):
    d = _dqn(hidden, rainbow_only)
    shapes = net.layer_shapes(18, hidden=hidden, rainbow_only=rainbow_only)
    sd = d.state_dict()
    assert set(sd) == set(shapes)
    for k, t in sd.items():
        assert tuple(t.shape) == tuple(shapes[k]), k
    hv, ha = d.fcnoisy_h_v, d.fcnoisy_h_a
    # [h_v | h_a] form one (2*hidden, 3136) operand in the parameter, gradient and epsilon arenas
    for name in ("weight_mu", "weight_sigma", "bias_mu", "bias_sigma"):
        pv, pa = getattr(hv, name), getattr(ha, name)
        assert pa.data_ptr() == pv.data_ptr() + 4 * pv.numel(), name
        assert pa.grad.data_ptr() == pv.grad.data_ptr() + 4 * pv.numel(), name
        assert pv.data.untyped_storage().data_ptr() == d._flat.untyped_storage().data_ptr()
    for name in ("weight_epsilon", "bias_epsilon"):
        ev, ea = getattr(hv, name), getattr(ha, name)
        assert ea.data_ptr() == ev.data_ptr() + 4 * ev.numel(), name
        assert ev.untyped_storage().data_ptr() == d._eps_flat.untyped_storage().data_ptr()
    assert tuple(d._w_eff_h.shape) == (2 * hidden, 3136)
    assert hv._w_eff.data_ptr() + 4 * hv._w_eff.numel() == ha._w_eff.data_ptr()


@pytest.mark.parametrize("hidden", [0, 64, 200, 500, 1152])
def test_unsupported_width_raises(hidden):
    with pytest.raises(ValueError, match="hidden_size"):
        _dqn(hidden)
    with pytest.raises(ValueError, match="hidden_size"):
        _dqn(hidden, rainbow_only=True)


def test_infeasible_dueling_shape_raises():
    from rainbow_iqn_apex_b200 import model
    for hidden in WIDTHS:               # every Atari action count fits at every width
        for a in range(1, 19):
            model.check_dueling_shape(hidden, a)
        assert model.dueling_smem_bytes(hidden, 31) <= model.SMEM_PER_BLOCK
    with pytest.raises(ValueError, match="action_space"):
        _dqn(1024, action_space=32)
    with pytest.raises(ValueError, match="action_space"):
        model.check_dueling_shape(256, 0)
    # the categorical head does not use the dueling kernels
    assert _dqn(256, rainbow_only=True, action_space=32).action_space == 32


def test_oracle_reproduces_hidden256_fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "iqn_hidden256.npz"))
    hidden, seed, batch, steps = int(g["hidden"]), int(g["seed"]), int(g["batch"]), int(g["steps"])
    assert hidden == 256
    cfg = cases.iqn_cfg(int(g["cfg_n_tau"]), int(g["cfg_n_tau_prime"]), int(g["cfg_n_quantile"]),
                        float(g["cfg_discount"]), int(g["cfg_n_step"]), float(g["cfg_kappa"]))
    params = net.make_params(seed, hidden=hidden)
    p_on, p_tg = net.to_torch(params, requires_grad=True), net.to_torch(params)
    adam = losses.Adam([k for k in p_on if net.is_trainable(k)], lr=5e-5, eps=3.125e-4)
    for s in range(steps):
        b = cases.make_batch(seed + 10 + s, batch, n_step=cfg["n_step"], discount=cfg["discount"])
        taus = tuple(torch.from_numpy(t) for t in cases.make_taus(seed + 20 + s, batch, cfg))
        noises = cases.make_noises(seed + 30 + s, hidden=hidden)
        keep = {}
        loss, grads = losses.learn_step(p_on, p_tg, adam, cases.batch_to_torch(b), torch.from_numpy(b["weights"]),
                                        noises, taus, cfg, keep=keep)
        assert np.allclose(loss.numpy(), g[f"loss_{s}"], rtol=1e-5, atol=0)
        assert np.array_equal(keep["a_star"].numpy(), g[f"a_star_{s}"])
        assert np.allclose(keep["theta"].detach().numpy(), g[f"theta_{s}"], rtol=1e-5, atol=1e-6)
        assert np.allclose(keep["target"].numpy(), g[f"target_{s}"], rtol=1e-5, atol=1e-6)
        for k, gr in grads.items():
            assert np.allclose(cases.tensor_digest(gr), g[f"grad_{s}_{k}"], rtol=2e-4, atol=1e-7), k
            assert np.allclose(cases.tensor_digest(p_on[k]), g[f"param_{s}_{k}"], rtol=1e-5, atol=1e-6), k
