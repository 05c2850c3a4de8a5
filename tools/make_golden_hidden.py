"""Golden fixture of the reference learner at a non-default hidden width (needs the reference checkout that
oracle/make_golden.py imports).

    python -m tools.make_golden_hidden            # writes tests/golden/iqn_hidden256.npz

The same harness as oracle/make_golden.py (stubs, injected noise and quantiles, the unmodified reference Learner),
with ``hidden_size`` passed through to the reference's args, the initial parameters and the injected noise factors.
It asserts that the oracle reproduces the reference at that width and stores the fixture in the layout of
golden_iqn's, plus ``hidden``.  The existing fixtures are not touched.
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import cases, losses, make_golden as mg, network as net  # noqa: E402


def build_ref_learner(params, batch, cfg, hidden):
    from rainbowiqn.learner import Learner
    inj = mg.Injector()
    for _ in range(2):                       # the constructor resets the noise of both nets once (model.py:23)
        inj.push_noise(net.make_noise(99, hidden=hidden))
    args = mg.ref_args(batch, cfg)
    args.hidden_size = hidden
    with inj:
        learner = Learner(args, 18, None)
    learner.online_net.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in params.items()})
    learner.update_target_net()
    learner.train()
    return learner


def golden_iqn_hidden(name, batch, cfg, steps, seed, hidden):
    params = net.make_params(seed, hidden=hidden)
    learner = build_ref_learner(params, batch, cfg, hidden)
    p_on = net.to_torch(params, requires_grad=True)
    p_tg = net.to_torch(params)
    adam = losses.Adam([k for k in p_on if net.is_trainable(k)], lr=5e-5, eps=3.125e-4)
    rec = {"batch": batch, "steps": steps, "seed": seed, "hidden": hidden, **{f"cfg_{k}": v for k, v in cfg.items()}}
    named = dict(learner.online_net.named_parameters())
    for s in range(steps):
        b = cases.make_batch(seed + 10 + s, batch, n_step=cfg["n_step"], discount=cfg["discount"])
        taus = cases.make_taus(seed + 20 + s, batch, cfg)
        noises = cases.make_noises(seed + 30 + s, hidden=hidden)
        tb = cases.batch_to_torch(b)
        w = torch.from_numpy(b["weights"])
        inj = mg.Injector()
        for nz in noises:
            inj.push_noise(nz)
        for t in taus:
            inj.push_tau(t)
        with inj:
            _, ref_loss = learner.learn(mg._FakeMem((np.arange(batch), tb[0], tb[1], tb[2], tb[3], tb[4], w)), None)
        assert not inj.noise_q and not inj.tau_q
        keep = {}
        o_loss, o_grads = losses.learn_step(p_on, p_tg, adam, tb, w, noises, tuple(torch.from_numpy(t) for t in taus), cfg,
                                            keep=keep)
        ref_loss = ref_loss.detach()
        err = float((ref_loss - o_loss).abs().max() / ref_loss.abs().max())
        print(f"[{name}] step {s}: loss max-rel-diff oracle vs reference = {err:.3e}")
        assert err < 1e-5, err
        for k, g in o_grads.items():
            rg = named[k].grad
            gerr = float((rg - g).abs().max() / (rg.abs().max() + 1e-30))
            assert gerr < 1e-4, (k, gerr)
        for k, t in learner.online_net.state_dict().items():
            if net.is_trainable(k):
                perr = float((t - p_on[k].detach()).abs().max())
                assert perr < 1e-6, (k, perr)
        rec[f"loss_{s}"] = ref_loss.numpy()
        rec[f"a_star_{s}"] = keep["a_star"].numpy()
        rec[f"target_{s}"] = keep["target"].numpy()
        rec[f"theta_{s}"] = keep["theta"].detach().numpy()
        for k in o_grads:
            rec[f"grad_{s}_{k}"] = cases.tensor_digest(named[k].grad)
            rec[f"param_{s}_{k}"] = cases.tensor_digest(learner.online_net.state_dict()[k])
    np.savez_compressed(os.path.join(mg.GOLD, name + ".npz"), **rec)


def main():
    mg._install_stubs()
    os.makedirs(mg.GOLD, exist_ok=True)
    torch.manual_seed(0)
    golden_iqn_hidden("iqn_hidden256", batch=32, cfg=cases.iqn_cfg(16, 12, 8), steps=2, seed=707, hidden=256)
    print("golden fixture written to", mg.GOLD)


if __name__ == "__main__":
    main()
