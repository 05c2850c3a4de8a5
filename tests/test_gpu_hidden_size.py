"""GPU: hidden widths other than 512 (every multiple of 128 up to 1024).  The z-layer + dueling kernels at each width
against float64, and the learner, the categorical head, the CUDA-graph step, the actor and checkpoints at 256 / 1024
against the CPU oracle and the reference fixture recorded at hidden 256."""
import os

import numpy as np
import pytest
import torch

from helpers import digest, load_params, make_args, rel_err
from oracle import actor as oactor, cases, losses, network as net

pytestmark = pytest.mark.gpu
WIDTHS = (128, 256, 384, 512, 640, 768, 896, 1024)
SMEM_PER_BLOCK = 227 * 1024


def _call():
    from rainbow_iqn_apex_b200._lib import call, ptr
    return call, ptr


def _args(dev, hidden, batch=32, cfg=None, **kw):
    args = make_args(dev, batch, cfg, **kw)
    args.hidden_size = hidden
    return args


def _loss_tol():
    from rainbow_iqn_apex_b200 import model
    return {"fp16": 5e-4, "bf16": 1e-3}.get(model.PRECISION["fwd"], 2e-4)


def _grad_tol():
    from rainbow_iqn_apex_b200 import model
    return 1e-3 if model.PRECISION["bwd"] in ("fp32", "bf16x3") else 1e-2


@pytest.fixture
def precision():
    from rainbow_iqn_apex_b200 import model
    old = dict(model.PRECISION)
    yield model.set_precision
    model.PRECISION.update(old)


class FakeMem:
    def __init__(self, sample):
        self.sample = sample

    def get_sample_from_mp_queue(self, q):
        return self.sample


def _dev_batch(b, dev):
    return (torch.from_numpy(b["states"]).to(dev), torch.from_numpy(b["actions"]).to(dev),
            torch.from_numpy(b["returns"]).to(dev), torch.from_numpy(b["next_states"]).to(dev),
            torch.from_numpy(b["nonterminals"]).to(dev))


def _qmajor(t, batch):
    nq = t.shape[0] // batch
    return t.reshape(batch, nq, -1).transpose(0, 1).reshape(batch * nq, -1)


# ----------------------------------------------------------------------------------------------- dueling kernels
@pytest.mark.parametrize("R,B", [(3000, 8), (8203, 1)])
@pytest.mark.parametrize("A", [6, 18])
@pytest.mark.parametrize("hidden", WIDTHS)
def test_dueling_fwd_widths(cuda_dev, hidden, A, R, B):
    """riqn_dueling_fwd at every width: the register kernel (ragged R < 4096) and the streamed kernel (R >= 4096) against
    float64; the streamed kernel is bit-identical to the register kernel run on < 4096-row slices."""
    call, ptr = _call()
    g = torch.Generator(device="cpu").manual_seed(hidden + 31 * A + R)
    h = torch.randn(R, 2 * hidden, generator=g).clamp_(min=0).to(cuda_dev)
    wz = (torch.randn(1 + A, hidden, generator=g) * 0.05).to(cuda_dev)
    bz = torch.randn(1 + A, generator=g).to(cuda_dev)
    q = torch.full((R, A), float("nan"), device=cuda_dev)
    call("riqn_dueling_fwd", R, B, hidden, A, ptr(h), ptr(wz), ptr(bz), ptr(q))
    h64, w64, b64 = h.double().cpu(), wz.double().cpu(), bz.double().cpu()
    v = h64[:, :hidden] @ w64[0] + b64[0]
    adv = h64[:, hidden:] @ w64[1:].t() + b64[1:]
    ref = (v[:, None] + adv - adv.mean(1, keepdim=True)).view(B, R // B, A).transpose(0, 1).reshape(R, A)
    assert rel_err(q.cpu().numpy(), ref.numpy()) < 5e-6
    if B == 1:
        parts = []
        for lo in range(0, R, 4000):
            n = min(4000, R - lo)
            qs = torch.empty(n, A, device=cuda_dev)
            call("riqn_dueling_fwd", n, 1, hidden, A, ptr(h[lo:lo + n]), ptr(wz), ptr(bz), ptr(qs))
            parts.append(qs)
        assert torch.equal(q, torch.cat(parts))


def _bwd_inputs(dev, hidden, A, R, B, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    h = torch.randn(R, 2 * hidden, generator=g).clamp_(min=0).to(dev)
    wz = (torch.randn(1 + A, hidden, generator=g) * 0.05).to(dev)
    dtheta = torch.randn(R, generator=g).to(dev)                       # quantile-major rows
    gscale = torch.rand(B, generator=g).add_(0.1).to(dev)
    actions = torch.randint(0, A, (B,), generator=g).to(dev)
    return h, wz, dtheta, gscale, actions


def _bwd_reference(h, wz, dtheta, gscale, gmul, actions, hidden, A, R, B):
    """float64 dh (R, 2*hidden) and dz (R, 32), rows sample-major like h."""
    Nq = R // B
    h64, w64 = h.double().cpu(), wz.double().cpu()
    gsm = (dtheta.double().cpu().view(Nq, B).t() * (gscale.double().cpu() * gmul)[:, None]).reshape(R)   # row b*Nq + q
    act = actions.cpu().repeat_interleave(Nq)
    wbar = w64[1:].mean(0)
    dh = torch.empty(R, 2 * hidden, dtype=torch.float64)
    dh[:, :hidden] = gsm[:, None] * w64[0][None]
    dh[:, hidden:] = gsm[:, None] * (w64[1 + act] - wbar[None])
    dh *= (h64 > 0)
    dz = torch.zeros(R, 32, dtype=torch.float64)
    dz[:, 0] = gsm
    onehot = torch.nn.functional.one_hot(act, A).double()
    dz[:, 1:1 + A] = gsm[:, None] * (onehot - 1.0 / A)
    return dh, dz


@pytest.mark.parametrize("A", [6, 18, 24])
@pytest.mark.parametrize("hidden", WIDTHS)
def test_dueling_bwd_widths(cuda_dev, hidden, A):
    """riqn_dueling_bwd and riqn_dueling_bwd_bf16 at every width: dh, dz and the column sums against float64; the bf16
    image equals the bf16 rounding of the fp32 dh; the transposed image, where it is requested and fits, is the exact
    transpose, and where it does not fit the call is refused."""
    call, ptr = _call()
    R, B, gmul = 1000, 8, 0.125
    h, wz, dtheta, gscale, actions = _bwd_inputs(cuda_dev, hidden, A, R, B, 7 * hidden + A)
    dh_ref, dz_ref = _bwd_reference(h, wz, dtheta, gscale, gmul, actions, hidden, A, R, B)
    dh = torch.full((R, 2 * hidden), float("nan"), device=cuda_dev)
    dz = torch.full((R, 32), float("nan"), device=cuda_dev)
    dz_bf = torch.empty(R, 32, dtype=torch.bfloat16, device=cuda_dev)
    call("riqn_dueling_bwd", R, B, hidden, A, ptr(h), ptr(wz), ptr(dtheta), ptr(gscale), gmul, ptr(actions), ptr(dh),
         ptr(dz), ptr(dz_bf))
    assert rel_err(dh.cpu().numpy(), dh_ref.numpy()) < 1e-6
    assert rel_err(dz.cpu().numpy(), dz_ref.numpy()) < 1e-6
    assert torch.equal(dz_bf, dz.to(torch.bfloat16))

    h_bf = h.to(torch.bfloat16)
    tile_fits = 4 * ((1 + A) * hidden + 3 * hidden) + 32 * 2 * hidden * 2 <= SMEM_PER_BLOCK
    for h_img in (None, h_bf):
        for want_t in (False, True):
            dh_hi = torch.empty(R, 2 * hidden, dtype=torch.bfloat16, device=cuda_dev)
            dh_hiT = torch.empty(2 * hidden, R, dtype=torch.bfloat16, device=cuda_dev) if want_t else None
            cs = torch.full((2 * hidden,), float("nan"), device=cuda_dev)
            dz2 = torch.full((R, 32), float("nan"), device=cuda_dev)
            dz2_bf = torch.empty(R, 32, dtype=torch.bfloat16, device=cuda_dev)
            args = ("riqn_dueling_bwd_bf16", R, B, hidden, A, ptr(h), ptr(h_img) if h_img is not None else None, ptr(wz),
                    ptr(dtheta), ptr(gscale), gmul, ptr(actions), ptr(dh_hi), ptr(dh_hiT) if want_t else None, ptr(cs),
                    ptr(dz2), ptr(dz2_bf))
            if want_t and not tile_fits:
                with pytest.raises(Exception, match="riqn_dueling_bwd_bf16"):
                    call(*args)
                continue
            call(*args)
            assert torch.equal(dh_hi, dh.to(torch.bfloat16))
            assert torch.equal(dz2, dz) and torch.equal(dz2_bf, dz_bf)
            assert rel_err(cs.cpu().numpy(), dh_ref.sum(0).numpy()) < 1e-5
            if want_t:
                assert torch.equal(dh_hiT, dh_hi.t())


# ----------------------------------------------------------------------------------------------- learner step
def _learner(dev, hidden, batch, cfg, params, rainbow_only=False):
    from rainbow_iqn_apex_b200 import Learner
    lr = Learner(_args(dev, hidden, batch, cfg, rainbow_only=rainbow_only), 18, None)
    load_params(lr.online_net, params)
    lr.update_target_net()
    lr.train()
    return lr


@pytest.mark.parametrize("mode", [None, ("fp32", "fp32")])
@pytest.mark.parametrize("hidden", [256, 1024])
def test_learn_vs_oracle(cuda_dev, precision, hidden, mode):
    """One Learner.learn (loss -> backward -> Adam) at hidden 256 / 1024 against the oracle, with injected noise and
    quantiles, in the default arithmetic and in fp32."""
    if mode is not None:
        precision(*mode)
    batch, cfg, seed = 32, cases.iqn_cfg(32, 32, 16), 4000 + hidden
    params = net.make_params(seed, hidden=hidden)
    lr = _learner(cuda_dev, hidden, batch, cfg, params)
    b = cases.make_batch(seed + 1, batch)
    taus = tuple(torch.from_numpy(t) for t in cases.make_taus(seed + 2, batch, cfg))
    noises = cases.make_noises(seed + 3, hidden=hidden)
    lr._inject = dict(noises=noises, taus=taus)
    lr._debug = {}
    w = torch.from_numpy(b["weights"])
    _, loss = lr.learn(FakeMem((np.arange(batch), *_dev_batch(b, cuda_dev), w.to(cuda_dev))), None)
    grads_gpu = {k: p.grad.detach().cpu().clone() for k, p in lr.online_net.named_parameters()}

    p_on, p_tg = net.to_torch(params, requires_grad=True), net.to_torch(params)
    adam = losses.Adam([k for k in p_on if net.is_trainable(k)], lr=5e-5, eps=3.125e-4)
    keep = {}
    o_loss, o_grads = losses.learn_step(p_on, p_tg, adam, cases.batch_to_torch(b), w, noises, taus, cfg, keep=keep)
    lg, lo = loss.cpu().numpy(), o_loss.numpy()
    bad = np.abs(lg - lo) / np.abs(lo) >= _loss_tol()
    if bad.any():       # only a double-DQN argmax on a numerical tie may move a transition's loss
        K = keep["q_sel"].shape[0] // batch
        qm = keep["q_sel"].reshape(K, batch, -1).mean(0).numpy()
        for i in np.where(bad)[0]:
            top = np.sort(qm[i])[-2:]
            assert top[1] - top[0] < 1e-3, (i, lg[i], lo[i])
        assert bad.sum() <= 1
    gk = lr._debug["keep"]
    hq = _qmajor(gk["h"], batch).cpu()
    flips = sum(int(((a.cpu() > 0) != (b_ > 0)).sum()) for a, b_ in
                ((gk["out"][0], keep["o1"]), (gk["out"][1], keep["o2"]), (gk["out"][2], keep["o3"]),
                 (hq[:, :hidden], keep["h_v"]), (hq[:, hidden:], keep["h_a"])))
    if bad.any():
        return
    named = dict(lr.online_net.named_parameters())
    for k, g_ref in o_grads.items():
        gg = grads_gpu[k]
        cos = float((gg * g_ref).sum() / (gg.norm() * g_ref.norm() + 1e-30))
        rel = float((gg - g_ref).norm() / (g_ref.norm() + 1e-30))
        if flips == 0:
            assert cos > 0.999 and rel < (3e-2 if mode is None else _grad_tol()), (k, cos, rel)
            assert np.allclose(named[k].detach().cpu().numpy(), p_on[k].detach().numpy(), rtol=0,
                               atol=1e-6 if _grad_tol() < 5e-3 else 5e-6), k
        else:
            assert cos > 0.98 and rel < 0.2, (k, cos, rel, flips)


def test_learn_matches_reference_golden_hidden256(cuda_dev, golden_dir):
    """Two Learner.learn calls at hidden 256 against the fixture recorded from the unmodified reference."""
    g = np.load(os.path.join(golden_dir, "iqn_hidden256.npz"))
    hidden, seed, batch, steps = int(g["hidden"]), int(g["seed"]), int(g["batch"]), int(g["steps"])
    cfg = cases.iqn_cfg(int(g["cfg_n_tau"]), int(g["cfg_n_tau_prime"]), int(g["cfg_n_quantile"]),
                        float(g["cfg_discount"]), int(g["cfg_n_step"]), float(g["cfg_kappa"]))
    params_np = net.make_params(seed, hidden=hidden)
    lr = _learner(cuda_dev, hidden, batch, cfg, params_np)
    p_or = net.to_torch(params_np)
    for s in range(steps):
        b = cases.make_batch(seed + 10 + s, batch, n_step=cfg["n_step"], discount=cfg["discount"])
        taus = tuple(torch.from_numpy(t) for t in cases.make_taus(seed + 20 + s, batch, cfg))
        lr._inject = dict(noises=cases.make_noises(seed + 30 + s, hidden=hidden), taus=taus)
        w = torch.from_numpy(b["weights"]).to(cuda_dev)
        lr._debug = {}
        _, loss = lr.learn(FakeMem((np.arange(batch), *_dev_batch(b, cuda_dev), w)), None)
        assert rel_err(loss.cpu().numpy(), g[f"loss_{s}"]) < _loss_tol()
        assert np.max(np.abs(loss.cpu().numpy() - g[f"loss_{s}"]) / np.abs(g[f"loss_{s}"])) < 1e-3
        # ReLU kinks that round to opposite sides of 0 on the CPU and the GPU move the upstream conv gradients
        keep_o = {}
        with torch.no_grad():
            losses.iqn_loss(p_or, net.to_torch(params_np), *cases.batch_to_torch(b), lr._inject["noises"],
                            lr._inject["taus"], **cfg, keep=keep_o)
        gk = lr._debug["keep"]
        fl = [int(((a.cpu() > 0) != (b_ > 0)).sum()) for a, b_ in ((gk["out"][0], keep_o["o1"]), (gk["out"][1], keep_o["o2"]),
                                                                   (gk["out"][2], keep_o["o3"]))]
        # a hidden-layer kink flip moves the data gradient of its row, hence every gradient below the head
        hq = _qmajor(gk["h"], batch).cpu()
        fh = sum(int(((a > 0) != (b_ > 0)).sum()) for a, b_ in ((hq[:, :hidden], keep_o["h_v"]), (hq[:, hidden:], keep_o["h_a"])))
        upstream = {"conv1": sum(fl) + fh, "conv2": fl[1] + fl[2] + fh, "conv3": fl[2] + fh, "iqn_fc": fh}
        for k, p in lr.online_net.named_parameters():
            gd, ref = digest(p.grad), g[f"grad_{s}_{k}"]
            nfl = upstream.get(k.split(".")[0], 0)
            gtol = _grad_tol() if nfl == 0 else min(0.25, 5e-2 * nfl)
            assert abs(gd[2] - ref[2]) <= gtol * ref[2] + 1e-9, (k, gd[:3], ref[:3], fl, fh)
            assert np.allclose(gd[3:], ref[3:], rtol=2 * gtol, atol=2 * gtol * ref[2] / np.sqrt(p.numel()) + 1e-9), (k, fl, fh)
            pd, pref = digest(p), g[f"param_{s}_{k}"]
            if nfl or _grad_tol() > 1e-3:
                assert np.allclose(pd[2:], pref[2:], rtol=1e-5, atol=5e-6), k
            else:
                assert np.allclose(pd, pref, rtol=1e-5, atol=1e-6), k
        for k, p in lr.online_net.named_parameters():
            p_or[k] = p.detach().cpu().clone()


def test_c51_learn_vs_oracle_hidden256(cuda_dev):
    """The categorical head (rainbow_only) at hidden 256: one Learner.learn against the oracle."""
    hidden, batch, seed = 256, 16, 8256
    params = net.make_params(seed, hidden=hidden, rainbow_only=True)
    lr = _learner(cuda_dev, hidden, batch, None, params, rainbow_only=True)
    b = cases.make_batch(seed + 1, batch)
    noises = cases.make_noises(seed + 3, hidden=hidden, rainbow_only=True)
    lr._inject = dict(noises=noises, taus=None)
    w = torch.from_numpy(b["weights"])
    _, loss = lr.learn(FakeMem((np.arange(batch), *_dev_batch(b, cuda_dev), w.to(cuda_dev))), None)
    p_on, p_tg = net.to_torch(params, requires_grad=True), net.to_torch(params)
    adam = losses.Adam([k for k in p_on if net.is_trainable(k)], lr=6.25e-5, eps=1.5e-4)
    ocfg = dict(atoms=51, v_min=-10.0, v_max=10.0, discount=0.99, n_step=3)
    o_loss, o_grads = losses.learn_step(p_on, p_tg, adam, cases.batch_to_torch(b), w, noises, None, ocfg, rainbow_only=True)
    assert np.max(np.abs(loss.cpu().numpy() - o_loss.numpy()) / np.abs(o_loss.numpy())) < 2e-4
    named = dict(lr.online_net.named_parameters())
    for k, gr in o_grads.items():
        gg = named[k].grad.cpu()
        cos = float((gg * gr).sum() / (gg.norm() * gr.norm() + 1e-30))
        assert cos > 0.999, (k, cos)


# ----------------------------------------------------------------------------------------------- graph, actor, checkpoint
def _graph_setup(dev, hidden, seed):
    from rainbow_iqn_apex_b200 import Learner, ReplayMemory
    torch.manual_seed(seed)
    args = _args(dev, hidden, 16, cases.iqn_cfg(16, 16, 8), nb_actor=1, actor_capacity=512)
    lr = Learner(args, 18, None)
    load_params(lr.online_net, net.make_params(5, hidden=hidden))
    lr.update_target_net()
    mem = ReplayMemory(args, None)
    rs = np.random.RandomState(1)
    n = 512
    mem.transitions.append_arrays(0, 0, np.arange(n) % 97, rs.randint(0, 256, (n, 84, 84)).astype(np.uint8),
                                  rs.randint(0, 18, n), rs.randint(-1, 2, n).astype(np.float32), rs.uniform(size=n) < 0.03,
                                  (rs.uniform(0.1, 1, n) ** 0.2).astype(np.float32))
    for obj, sd in ((lr.online_net, 11), (lr.target_net, 12), (mem.transitions, 13)):
        obj._rng_seed = sd
    return lr, mem


def test_graph_replay_matches_eager_hidden256(cuda_dev):
    from rainbow_iqn_apex_b200.dynstate import DynState
    a, mem_a = _graph_setup(cuda_dev, 256, 0)
    b, mem_b = _graph_setup(cuda_dev, 256, 0)
    a.enable_cuda_graph(mem_a, warmup=2)
    b._dyn = DynState(cuda_dev)
    b._attach_dyn(mem_b, True)

    def eager_step():
        nss, sbc = b.optimiser.bias_corrections(b.optimiser._step + 1)
        b._dyn.write(nss, sbc, mem_b.transitions.get_current_capacity(), mem_b.priority_weight)
        return b._step_body(mem_b)

    for _ in range(2):
        eager_step()
    b._dyn.epoch += 1
    losses_a = []
    for _ in range(3):
        ia, la = a.learn_and_update(mem_a)
        ib, lb = eager_step()
        assert torch.equal(ia, ib)
        assert torch.allclose(la, lb, rtol=2e-3, atol=1e-6)
        losses_a.append(la.clone())
    assert a.optimiser._step == b.optimiser._step == 5
    d = (a.online_net._flat - b.online_net._flat).abs()
    assert float(d.max()) <= 3 * 5e-5 + 1e-6
    assert int((d > 1e-5).sum()) <= 5 * 3136
    assert not torch.equal(losses_a[0], losses_a[1]) and torch.isfinite(torch.stack(losses_a)).all()


def test_actor_hidden256_vs_oracle(cuda_dev):
    """Actor.act_batch and Actor.compute_priorities at hidden 256 against the oracle."""
    from rainbow_iqn_apex_b200 import Actor
    hidden, E, seed, cfg = 256, 24, 9256, cases.iqn_cfg(16, 16, 8)
    params = net.make_params(seed, hidden=hidden)
    actor = Actor(_args(cuda_dev, hidden, 8, cfg, actor_capacity=64), 18, None)
    load_params(actor.online_net, params)
    actor.update_target_net()
    actor.train()
    noise = net.make_noise(seed + 1, hidden=hidden)
    actor.online_net.reset_noise(noise)
    rs = np.random.RandomState(seed)
    states = rs.randint(0, 256, (E, 4, 84, 84)).astype(np.uint8)
    K = cfg["n_quantile"]
    tau = rs.uniform(0, 1, (K * E, 1)).astype(np.float32)
    actor._inject_act_tau = torch.from_numpy(tau)
    a = actor.act_batch(torch.from_numpy(states).to(cuda_dev)).cpu().numpy()
    actor._inject_act_tau = torch.from_numpy(tau)
    qm = actor.act_batch_values(torch.from_numpy(states).to(cuda_dev)).cpu().numpy()
    with torch.no_grad():
        q = net.dqn_forward_iqn(net.apply_noise(net.to_torch(params), noise), torch.from_numpy(states).float().div_(255), K,
                                torch.from_numpy(tau))
    qo = q.reshape(K, E, 18).mean(0).numpy()
    assert rel_err(qm, qo) < 1e-3
    ao = qo.argmax(1)
    for e in np.where(a != ao)[0]:
        assert abs(qo[e, ao[e]] - qo[e, a[e]]) < 1e-4
    assert (a != ao).sum() <= 1
    # compute_priorities over one synthetic buffer (an episode end in the middle), one injection per chunk
    L, bs = 22, 8
    frames = rs.randint(0, 256, (L + 3, 84, 84)).astype(np.uint8)
    tab_state = [frames[i] for i in range(len(frames))]
    tab_action = [int(x) for x in rs.randint(0, 18, L)]
    tab_reward = [float(x) for x in rs.randint(-1, 2, L)]
    tab_nonterminal = [True] * L
    tab_nonterminal[L // 2] = False
    n_tr = L - cfg["n_step"]
    chunks = [(lo, min(lo + bs, n_tr)) for lo in range(0, n_tr, bs)]
    noises = [cases.make_noises(seed + 100 + c, hidden=hidden) for c in range(len(chunks))]
    taus = [tuple(torch.from_numpy(rs.uniform(0, 1, (nq * (hi - lo), 1)).astype(np.float32))
                  for nq in (K, cfg["n_tau_prime"], cfg["n_tau"])) for lo, hi in chunks]
    actor._inject = [dict(noises=noises[c], taus=taus[c]) for c in range(len(chunks))]
    pri = actor.compute_priorities(tab_state, tab_action, tab_reward, tab_nonterminal, 0.2)
    pri_or = oactor.compute_priorities(net.to_torch(params), net.to_torch(params), tab_state, tab_action, tab_reward,
                                       tab_nonterminal, 0.2, noises, taus, cfg, bs)
    assert pri.shape == pri_or.shape and not actor._inject
    assert np.max(np.abs(pri - pri_or) / np.abs(pri_or)) < 1e-3


def test_checkpoint_roundtrip_hidden256(cuda_dev, tmp_path):
    """Agent.save at hidden 256, then a new Agent from that checkpoint (args.model): identical parameters and q."""
    from rainbow_iqn_apex_b200 import Agent
    hidden, cfg = 256, cases.iqn_cfg(8, 8, 4)
    ag = Agent(_args(cuda_dev, hidden, 4, cfg), 18, None)
    load_params(ag.online_net, net.make_params(43, hidden=hidden))
    ag.save(str(tmp_path), 1, 2, "ckpt.pth")
    ck = torch.load(os.path.join(str(tmp_path), "ckpt.pth"), map_location="cpu")
    assert {k: tuple(v.shape) for k, v in ck["model_state_dict"].items()} == \
        {k: tuple(s) for k, s in net.layer_shapes(18, hidden=hidden).items()}
    args = _args(cuda_dev, hidden, 4, cfg)
    args.model = os.path.join(str(tmp_path), "ckpt.pth")
    ag2 = Agent(args, 18, None)
    assert torch.equal(ag2.online_net._flat, ag.online_net._flat)
    x = torch.from_numpy(cases.make_batch(44, 4)["states"]).to(cuda_dev)
    tau = torch.rand(8 * 4, 1, generator=torch.Generator().manual_seed(45))
    with torch.no_grad():
        qa, _ = ag.online_net(x, 8, tau=tau)
        qb, _ = ag2.online_net(x, 8, tau=tau)
    assert qa.shape == (32, 18) and torch.equal(qa, qb)
    # a checkpoint of one width does not load into a network of another
    args.hidden_size = 512
    with pytest.raises(RuntimeError):
        Agent(args, 18, None)
