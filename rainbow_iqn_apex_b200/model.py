"""DQN / NoisyLinear with the reference's API and state_dict keys, computed by libriqn_b200.so.

Mirrors ``rainbowiqn/model.py`` of the reference (NoisyLinear :9-53, DQN :56-162):
same constructor arguments, same parameter / buffer names and shapes
(``conv{1,2,3}.{weight,bias}``, ``iqn_fc.{weight,bias}``,
``fcnoisy_{h_v,h_a,z_v,z_a}.{weight_mu,weight_sigma,bias_mu,bias_sigma,weight_epsilon,bias_epsilon}``),
same ``forward(x, num_quantiles)`` -> ``(q (Nq*B, A), quantiles (Nq*B, 1))`` row convention
(row = quantile * B + sample) and same ``reset_noise()`` semantics.

B200-native layout: all trainable parameters live in ONE flat fp32 arena in HBM (gradients and the
Adam moments in matching arenas), ordered so that fcnoisy_h_v|fcnoisy_h_a form a single
(2*hidden, 3136) operand and fcnoisy_z_v|fcnoisy_z_a a single (1+A, hidden) operand.  The nn.Parameters
are views of the arena, so torch's state_dict / load_state_dict / checkpoints keep working while the
optimiser and the gradient all-reduce touch one contiguous buffer.

Supported widths: ``hidden_size`` is any multiple of 128 up to 1024 (``HIDDEN_SIZES``).  The z-layer + dueling kernels
are instantiated once per width; the head products take the width at run time.  Other widths raise ValueError, and so
does an IQN action space the dueling kernels cannot hold (``check_dueling_shape``).

There is no PyTorch fallback: every tensor operation below is a C-ABI call (include/riqn_b200.h).
"""
import math
import os
import weakref

import torch
from torch import nn

from . import _lib
from ._lib import ConvGeom, NoisyLayer, SplitJob, call, ptr

FEAT = 3136
# Philox stream ids: CUDA-graph steps use (static per-step index + the device-side rng_offset = 64 * epoch); eager calls count
# on the host.  The eager counters live in their own half of the id space so that the two can never reuse a stream.
_EAGER_STREAMS = 1 << 39
_ALIGN = 64  # floats; arena groups start on 256-byte boundaries

# Arithmetic of the hidden NoisyLinear products (x W^T, dh W, dh^T x -- 91% of the step's FLOPs):
#   "bf16x3": tcgen05 tensor cores, every operand split into bf16 hi + lo, 3 MMAs per k-step (fp32-faithful)
#   "bf16"  : tcgen05 tensor cores, operands rounded to bf16 once, fp32 accumulation in TMEM
#   "fp16"  : (forward only) ONE tcgen05 pass on fp16 images of x and W (11-bit significands: the error of a tf32 product
#             at the bf16 rate; activations / weights of this network sit far inside the fp16 range).  The small products
#             (conv trunk, quantile embedding: 5% of the FLOPs) keep the split-bf16 x3 arithmetic.
#   "fp32"  : CUDA-core fp32 GEMM (gemm_simt.cu), the cross-check path
PRECISION = {"fwd": os.environ.get("RIQN_FWD_PRECISION", "fp16"), "bwd": os.environ.get("RIQN_BWD_PRECISION", "bf16")}
WGRAD_SPLIT_K = int(os.environ.get("RIQN_WGRAD_SPLIT_K", "4"))
_NO_STRIP = os.environ.get("RIQN_NO_STRIP_CONV", "0") == "1"      # fall back to the explicit-im2col forward

# Widths of the two hidden NoisyLinear layers with z-layer + dueling kernels: 2*hidden is then a multiple of 256 (whole
# head-product n-tiles) and every lane of the dueling kernels owns whole float4 / 8-wide bf16 chunks.
HIDDEN_SIZES = tuple(range(128, 1025, 128))
MAX_DUELING_ACTIONS = 31          # the dueling kernels keep one advantage per lane (lane 0 holds the value)
SMEM_PER_BLOCK = 227 * 1024       # opt-in dynamic shared memory per block on sm_100a


def dueling_smem_bytes(hidden, action_space):
    """Largest dynamic shared memory the IQN head's z-layer + dueling kernels need for (hidden, A) on the learner path:
    the (1+A, hidden) z-weights, plus the advantage column means and the 2*hidden column sums of the backward."""
    return 4 * max((1 + action_space) * hidden,             # riqn_dueling_fwd
                   (1 + action_space) * hidden + hidden,    # riqn_dueling_bwd
                   (1 + action_space) * hidden + 3 * hidden)  # riqn_dueling_bwd_bf16 (no transposed image)


def check_dueling_shape(hidden, action_space):
    """Raise ValueError unless the IQN head's kernels run at this (hidden, A)."""
    if hidden not in HIDDEN_SIZES:
        raise ValueError(f"hidden_size={hidden} is not supported: the sm_100a kernels take hidden_size in {HIDDEN_SIZES} "
                         "(a multiple of 128 up to 1024)")
    if not 1 <= action_space <= MAX_DUELING_ACTIONS:
        raise ValueError(f"action_space={action_space} is not supported by the IQN dueling kernels (1..{MAX_DUELING_ACTIONS})")
    need = dueling_smem_bytes(hidden, action_space)
    if need > SMEM_PER_BLOCK:
        raise ValueError(f"hidden_size={hidden} with action_space={action_space} needs {need} bytes of shared memory per "
                         f"block in the dueling kernels; the limit is {SMEM_PER_BLOCK}")


def set_precision(fwd=None, bwd=None):
    for k, v in (("fwd", fwd), ("bwd", bwd)):
        if v is not None:
            if v not in ("bf16x3", "bf16", "fp32") + (("fp16",) if k == "fwd" else ()):
                raise ValueError(v)
            PRECISION[k] = v
    if PRECISION["fwd"] == "fp16" and PRECISION["bwd"] != "bf16":
        raise ValueError("the fp16 forward pairs with the bf16 backward (it reads the bf16 images written beside the fp16 ones)")


def _small_x3():
    """Split-bf16 x3 arithmetic for the conv trunk and the embedding product (both memory-bound)."""
    return PRECISION["fwd"] in ("bf16x3", "fp16")


class NoisyLinear(nn.Module):
    """Factorised-noise linear layer (reference model.py:9-53)."""

    def __init__(self, in_features, out_features, std_init, disable_cuda=False):
        super().__init__()
        self.disable_cuda = disable_cuda
        self.in_features = in_features
        self.out_features = out_features
        self.std_init = std_init
        self.weight_mu = nn.Parameter(torch.empty(out_features, in_features))
        self.weight_sigma = nn.Parameter(torch.empty(out_features, in_features))
        self.register_buffer("weight_epsilon", torch.zeros(out_features, in_features))
        self.bias_mu = nn.Parameter(torch.empty(out_features))
        self.bias_sigma = nn.Parameter(torch.empty(out_features))
        self.register_buffer("bias_epsilon", torch.zeros(out_features))
        # scratch for the factor vectors f(eps_in), f(eps_out) and the composed weights (set by DQN)
        self._eps_in = None
        self._eps_out = None
        self._w_eff = None
        self._b_eff = None
        self._noise_calls = 0
        self._calls_in_step = 0
        self._dyn = None    # DynState in CUDA-graph mode (set by Learner.enable_cuda_graph)
        self._layer_id = 0  # distinct Philox streams per layer (set by DQN)
        self.reset_parameters()

    def reset_parameters(self):
        """model.py:25-30"""
        mu_range = 1 / math.sqrt(self.in_features)
        self.weight_mu.data.uniform_(-mu_range, mu_range)
        self.weight_sigma.data.fill_(self.std_init / math.sqrt(self.in_features))
        self.bias_mu.data.uniform_(-mu_range, mu_range)
        self.bias_sigma.data.fill_(self.std_init / math.sqrt(self.out_features))

    def _ensure_scratch(self):
        dev = self.weight_mu.device
        if self._eps_in is None or self._eps_in.device != dev:
            self._eps_in = torch.empty(self.in_features, device=dev)
            self._eps_out = torch.empty(self.out_features, device=dev)
        if self._w_eff is None or self._w_eff.device != dev:
            self._w_eff = torch.empty(self.out_features, self.in_features, device=dev)
            self._b_eff = torch.empty(self.out_features, device=dev)

    def reset_noise(self, eps_in=None, eps_out=None, seed=None):
        """model.py:39-43.  ``eps_in``/``eps_out`` inject already-scaled factor vectors (parity runs);
        otherwise they are drawn on the device (Philox) as f(N(0,1)), f(x)=sign(x)sqrt|x| (model.py:32-37)."""
        self._ensure_scratch()
        if eps_in is None:
            if seed is None:
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            dyn = self._dyn
            # graph mode: static per-step index (the device-side rng_offset advances the stream every step)
            idx = self._calls_in_step if dyn is not None else self._noise_calls
            base = (self._layer_id << 40) + 2 * idx + (0 if dyn is not None else _EAGER_STREAMS)
            call("riqn_noisy_sample", self.in_features, seed, base, ptr(self._eps_in), dyn.ptr() if dyn else None)
            call("riqn_noisy_sample", self.out_features, seed, base + 1, ptr(self._eps_out), dyn.ptr() if dyn else None)
            self._noise_calls += 1
            self._calls_in_step += 1
        else:
            self._eps_in.copy_(eps_in)
            self._eps_out.copy_(eps_out)
        self._compose(resample=True)

    def _compose(self, resample=False):
        self._ensure_scratch()
        call("riqn_noisy_compose", self.out_features, self.in_features, ptr(self.weight_mu), ptr(self.weight_sigma),
             ptr(self.weight_epsilon), ptr(self._eps_in) if resample else None,
             ptr(self._eps_out) if resample else None, ptr(self.bias_mu), ptr(self.bias_sigma),
             ptr(self.bias_epsilon), ptr(self._w_eff), ptr(self._b_eff), 1 if self.training else 0)

    def forward(self, input):
        """model.py:45-53 (inference helper; the learner path goes through DQN's fused ops)."""
        self._compose()
        x = input.contiguous().float()
        out = torch.empty(x.shape[0], self.out_features, device=x.device)
        call("riqn_gemm_f32", x.shape[0], self.out_features, self.in_features, ptr(x), self.in_features, 1,
             ptr(self._w_eff), self.in_features, 1, ptr(out), self.out_features)
        return out + self._b_eff


def _strip_perm(cin, k, stride, first):
    """Column permutation of a (Cout, Cin*k*k) weight for the strip convolution: new index (dy, dx, within-block) ->
    original index c*k*k + kh*k + kw, with kh = stride*dy + iy, kw = stride*dx + ix.  Within a block the first layer
    (uint8 frames, riqn_s2d_u8) is ordered (c, iy, ix); later layers (written by the previous layer's epilogue) are
    ordered (iy, ix, c)."""
    t = k // stride
    idx = []
    for dy in range(t):
        for dx in range(t):
            if first:
                order = [(c, iy, ix) for c in range(cin) for iy in range(stride) for ix in range(stride)]
            else:
                order = [(c, iy, ix) for iy in range(stride) for ix in range(stride) for c in range(cin)]
            idx += [c * k * k + (stride * dy + iy) * k + (stride * dx + ix) for c, iy, ix in order]
    return torch.tensor(idx, dtype=torch.long)


def _geom(batch, cin, h, cout, k, stride, pad, in_bstride=None):
    oh = (h + 2 * pad - k) // stride + 1
    return ConvGeom(batch, cin, h, h, cout, k, k, stride, pad, oh, oh, in_bstride if in_bstride else cin * h * h)


class DQN(nn.Module):
    """Reference model.py:56-162 (IQN branch; the C51 branch lives in c51.py).  ``args.hidden_size`` must be in
    HIDDEN_SIZES; the IQN head also needs ``check_dueling_shape(hidden_size, action_space)`` to pass."""

    def __init__(self, args, action_space):
        super().__init__()
        self.rainbow_only = args.rainbow_only
        self.action_space = action_space
        self.device = args.device
        self.disable_cuda = args.disable_cuda
        self.history = args.history_length
        self.hidden = args.hidden_size
        if self.hidden not in HIDDEN_SIZES:
            raise ValueError(f"hidden_size={self.hidden} is not supported: the sm_100a kernels take hidden_size in "
                             f"{HIDDEN_SIZES} (a multiple of 128 up to 1024)")
        if not self.rainbow_only:
            check_dueling_shape(self.hidden, action_space)
        self.conv1 = nn.Conv2d(args.history_length, 32, 8, stride=4, padding=1)
        self.conv2 = nn.Conv2d(32, 64, 4, stride=2)
        self.conv3 = nn.Conv2d(64, 64, 3)
        if self.rainbow_only:
            self.atoms = args.atoms
            self._v_min, self._v_max = args.V_min, args.V_max
            zv, za = self.atoms, action_space * self.atoms
        else:
            self.quantile_embedding_dim = args.quantile_embedding_dim
            self.iqn_fc = nn.Linear(self.quantile_embedding_dim, FEAT)
            zv, za = 1, action_space
        kw = dict(std_init=args.noisy_std, disable_cuda=args.disable_cuda)
        # "fcnoisy" in the name marks the noisy layers (model.py:159-162)
        self.fcnoisy_h_v = NoisyLinear(FEAT, args.hidden_size, **kw)
        self.fcnoisy_h_a = NoisyLinear(FEAT, args.hidden_size, **kw)
        self.fcnoisy_z_v = NoisyLinear(args.hidden_size, zv, **kw)
        self.fcnoisy_z_a = NoisyLinear(args.hidden_size, za, **kw)
        for i, m in enumerate((self.fcnoisy_h_v, self.fcnoisy_h_a, self.fcnoisy_z_v, self.fcnoisy_z_a)):
            m._layer_id = i + 1
        self._tau_calls = 0
        self._tau_in_step = 0
        self._dyn = None
        self._tau_stream_offset = 0   # rank-private quantile stream under data parallelism
        self._rng_seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        self._flatten()
        # anything that rewrites the noise-free weights must invalidate their cached bf16 operand images
        self.register_load_state_dict_post_hook(lambda module, _incompatible: setattr(module, "_static_ops_dirty", True))
        if self._flat.is_cuda:
            self.reset_noise()

    # ------------------------------------------------------------------ arenas
    def _param_groups_in_arena_order(self):
        g = [[self.conv1.weight], [self.conv1.bias], [self.conv2.weight], [self.conv2.bias],
             [self.conv3.weight], [self.conv3.bias]]
        if not self.rainbow_only:
            g += [[self.iqn_fc.weight], [self.iqn_fc.bias]]
        hv, ha, zv, za = self.fcnoisy_h_v, self.fcnoisy_h_a, self.fcnoisy_z_v, self.fcnoisy_z_a
        g += [[hv.weight_mu, ha.weight_mu], [hv.weight_sigma, ha.weight_sigma],
              [hv.bias_mu, ha.bias_mu], [hv.bias_sigma, ha.bias_sigma],
              [zv.weight_mu, za.weight_mu], [zv.weight_sigma, za.weight_sigma],
              [zv.bias_mu, za.bias_mu], [zv.bias_sigma, za.bias_sigma]]
        return g

    def _flatten(self):
        """(Re)build the flat parameter / gradient / epsilon arenas on the parameters' current device."""
        groups = self._param_groups_in_arena_order()
        dev = groups[0][0].device
        total = 0
        offsets = []
        for grp in groups:
            total = (total + _ALIGN - 1) // _ALIGN * _ALIGN
            for p in grp:
                offsets.append(total)
                total += p.numel()
        total = (total + _ALIGN - 1) // _ALIGN * _ALIGN
        flat = torch.zeros(total, device=dev, dtype=torch.float32)
        flat_grad = torch.zeros(total, device=dev, dtype=torch.float32)
        i = 0
        self._offsets = {}
        for grp in groups:
            for p in grp:
                off, n = offsets[i], p.numel()
                flat[off:off + n].copy_(p.data.reshape(-1).float())
                p.data = flat[off:off + n].view(p.shape)
                p.grad = flat_grad[off:off + n].view(p.shape)
                self._offsets[id(p)] = off
                p._riqn_owner = weakref.ref(self)
                p._riqn_offset = off
                i += 1
        self._flat, self._flat_grad = flat, flat_grad
        self._static_ops_dirty = True
        # epsilon arena: [h_v.weight_epsilon | h_a.weight_epsilon], h bias eps, [z_v | z_a] weight eps, z bias eps
        hv, ha, zv, za = self.fcnoisy_h_v, self.fcnoisy_h_a, self.fcnoisy_z_v, self.fcnoisy_z_a
        eg = [[(hv, "weight_epsilon"), (ha, "weight_epsilon")], [(hv, "bias_epsilon"), (ha, "bias_epsilon")],
              [(zv, "weight_epsilon"), (za, "weight_epsilon")], [(zv, "bias_epsilon"), (za, "bias_epsilon")]]
        etotal, eoffs = 0, []
        for grp in eg:
            etotal = (etotal + _ALIGN - 1) // _ALIGN * _ALIGN
            for m, name in grp:
                eoffs.append(etotal)
                etotal += m._buffers[name].numel()
        eflat = torch.zeros(etotal + _ALIGN, device=dev, dtype=torch.float32)
        i = 0
        for grp in eg:
            for m, name in grp:
                old = m._buffers[name]
                n = old.numel()
                eflat[eoffs[i]:eoffs[i] + n].copy_(old.reshape(-1).float())
                m._buffers[name] = eflat[eoffs[i]:eoffs[i] + n].view(old.shape)
                i += 1
        self._eps_flat = eflat
        # composed (effective) weights, concatenated like the arenas
        hid = self.hidden
        nz = zv.out_features + za.out_features
        self._w_eff_h = torch.empty(2 * hid, FEAT, device=dev)
        self._b_eff_h = torch.empty(2 * hid, device=dev)
        self._w_eff_z = torch.empty(nz, hid, device=dev)
        self._b_eff_z = torch.empty(nz, device=dev)
        hv._w_eff, ha._w_eff = self._w_eff_h[:hid], self._w_eff_h[hid:]
        hv._b_eff, ha._b_eff = self._b_eff_h[:hid], self._b_eff_h[hid:]
        zv._w_eff, za._w_eff = self._w_eff_z[:zv.out_features], self._w_eff_z[zv.out_features:]
        zv._b_eff, za._b_eff = self._b_eff_z[:zv.out_features], self._b_eff_z[zv.out_features:]
        for m in (hv, ha, zv, za):
            m._eps_in = torch.empty(m.in_features, device=dev)
            m._eps_out = torch.empty(m.out_features, device=dev)

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._flatten()
        if self._flat.is_cuda:
            self.reset_noise()  # NoisyLinear.__init__ resets noise in the reference (model.py:23)
        return out

    def zero_grad(self, set_to_none=False):
        """One memset over the gradient arena; the .grad views stay bound (learner.py:22)."""
        if self._flat_grad.is_cuda:
            call("riqn_zero_f32", ptr(self._flat_grad), self._flat_grad.numel())
        else:                       # CPU arenas exist only for the host-logic tests (gloo); nothing computes there
            self._flat_grad.zero_()
        for grp in self._param_groups_in_arena_order():
            for p in grp:
                if p.grad is None or p.grad.data_ptr() != self._flat_grad.data_ptr() + 4 * self._offsets[id(p)]:
                    off = self._offsets[id(p)]
                    p.grad = self._flat_grad[off:off + p.numel()].view(p.shape)

    def grad_view(self, p):
        off = self._offsets[id(p)]
        return self._flat_grad[off:off + p.numel()].view(p.shape)

    def noisy_layers(self):
        return [(n, m) for n, m in self.named_children() if "fcnoisy" in n]

    # ------------------------------------------------------------------ noise
    def reset_noise(self, noise=None):
        """model.py:159-162.  ``noise``: optional {layer_name: (f(eps_in), f(eps_out))} injection.
        All NoisyLinear layers are redrawn and recomposed by ONE riqn_noisy_reset_net call (two launches)."""
        self._noise_version = getattr(self, "_noise_version", 0) + 1     # backward passes check it: they read the LIVE weights
        layers = self.noisy_layers()
        if not self._flat.is_cuda or any(m.in_features % 4 for _, m in layers):
            for name, module in layers:
                if noise is not None:
                    e_in, e_out = noise[name]
                    module.reset_noise(e_in.to(self._flat.device), e_out.to(self._flat.device))
                else:
                    module.reset_noise(seed=self._rng_seed)
            self._refresh_tc_operands()
            return
        desc = self._noisy_desc()
        for k, (name, m) in enumerate(layers):
            if noise is not None:
                e_in, e_out = noise[name]
                m._eps_in.copy_(e_in)
                m._eps_out.copy_(e_out)
            else:
                # graph mode: static per-step index (the device-side rng_offset advances the stream every step)
                idx = m._calls_in_step if m._dyn is not None else m._noise_calls
                base = (m._layer_id << 40) + 2 * idx + (0 if m._dyn is not None else _EAGER_STREAMS)
                desc[k].stream_in, desc[k].stream_out = base, base + 1
                m._noise_calls += 1
                m._calls_in_step += 1
        dyn = layers[0][1]._dyn
        seed = self._rng_seed
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        call("riqn_noisy_reset_net", len(layers), desc, seed, 0 if noise is not None else 1, 1 if self.training else 0,
             dyn.ptr() if (dyn is not None and noise is None) else None)
        self._refresh_tc_operands(h_done=self._fuse_h_images())

    def _noisy_desc(self):
        """Cached riqn_noisy_layer[] for riqn_noisy_reset_net (all pointers are static arena / scratch addresses)."""
        layers = self.noisy_layers()
        fuse = self._fuse_h_images()
        w_hi = getattr(self, "_w_hi", None) if fuse else None
        f16 = PRECISION["fwd"] == "fp16"
        key = tuple(m.weight_mu.data_ptr() for _, m in layers) + (self._flat.data_ptr(), w_hi.data_ptr() if fuse else 0, f16)
        if getattr(self, "_noisy_desc_key", None) != key:
            arr = (NoisyLayer * len(layers))()
            for k, (name, m) in enumerate(layers):
                if fuse and name in ("fcnoisy_h_v", "fcnoisy_h_a"):
                    # the composed hidden-layer weights leave the compose kernel as bf16 (hi, lo) images as well
                    row0 = 0 if name == "fcnoisy_h_v" else self.hidden
                    arr[k].w_hi = self._w_hi.data_ptr() + row0 * FEAT * 2
                    arr[k].w_lo = self._w_lo.data_ptr() + row0 * FEAT * 2     # fp16 mode: bf16(w), the dgrad operand
                    arr[k].w_fp16 = 1 if f16 else 0
                m._ensure_scratch()
                d = arr[k]
                d.out_features, d.in_features = m.out_features, m.in_features
                d.weight_mu, d.weight_sigma, d.weight_epsilon = ptr(m.weight_mu), ptr(m.weight_sigma), ptr(m.weight_epsilon)
                d.bias_mu, d.bias_sigma, d.bias_epsilon = ptr(m.bias_mu), ptr(m.bias_sigma), ptr(m.bias_epsilon)
                d.eps_in, d.eps_out, d.w_eff, d.b_eff = ptr(m._eps_in), ptr(m._eps_out), ptr(m._w_eff), ptr(m._b_eff)
            self._noisy_desc_arr, self._noisy_desc_key = arr, key
        return self._noisy_desc_arr

    def _fuse_h_images(self):
        """True when reset_noise() can let the compose kernel write the bf16 images of the hidden-layer weights (every
        mode whose backward reads W itself; the transposed images of the other modes still come from riqn_split_bf16)."""
        if not self._flat.is_cuda or PRECISION["fwd"] == "fp32" or PRECISION["bwd"] != "bf16":
            return False
        self._ensure_tc_buffers()
        return True

    def compose_weights(self):
        """Recompute the effective weights from the stored epsilons (after load_state_dict / optimiser steps)."""
        for _, module in self.noisy_layers():
            module._compose()
        self._refresh_tc_operands(force=True)

    def _ensure_tc_buffers(self):
        """Allocate the bf16 operand images once per device."""
        dev = self._flat.device
        if getattr(self, "_w_hi", None) is None or self._w_hi.device != dev:
            n = 2 * self.hidden
            mk = lambda *sh: torch.empty(*sh, dtype=torch.bfloat16, device=dev)
            self._w_hi, self._w_lo = mk(n, FEAT), mk(n, FEAT)
            self._w_hiT, self._w_loT = mk(FEAT, n), mk(FEAT, n)
            self._conv_ops = {}
            self._static_ops_dirty = True
            for name, conv in (("conv1", self.conv1), ("conv2", self.conv2), ("conv3", self.conv3)):
                co, k = conv.weight.shape[0], conv.weight[0].numel()
                self._conv_ops[name] = (mk(co, k), mk(co, k), mk(k, co))
            k1 = self.conv1.weight[0].numel()
            self._conv1_px_ops = (mk(32, k1), mk(32, k1))      # bf16 hi / lo of conv1.weight / 255 (uint8 ingest)
            if not self.rainbow_only:
                self._iqn_ops = (mk(FEAT, self.quantile_embedding_dim), mk(FEAT, self.quantile_embedding_dim))

    def _refresh_tc_operands(self, force=False, h_done=False):
        """bf16 (hi, lo) images of the composed hidden-layer weights for the tcgen05 path: (2*hid, 3136) K-major for
        the forward product and the transposed (3136, 2*hid) copy the data-gradient product consumes.  The images of
        the noise-free weights (convolutions, iqn_fc) are only rebuilt when those weights may have changed: after an
        optimiser step (optim.Adam marks the owner), after compose_weights() (``force``), or on first use."""
        if (PRECISION["fwd"] == "fp32" and PRECISION["bwd"] == "fp32") or not self._flat.is_cuda:
            return
        self._ensure_tc_buffers()
        dev = self._flat.device
        need_t = PRECISION["bwd"] != "bf16" or PRECISION["fwd"] == "fp32"   # bf16 backward reads W itself (MN-major operand)
        if not h_done:
            f16 = PRECISION["fwd"] == "fp16"
            call("riqn_split_bf16", 2 * self.hidden, FEAT, ptr(self._w_eff_h), ptr(self._w_hi), ptr(self._w_lo),
                 ptr(self._w_hiT) if need_t else None, ptr(self._w_loT) if need_t else None, 1 if f16 else 0)
        if not (force or getattr(self, "_static_ops_dirty", True)):
            return
        self._static_ops_dirty = False
        # strip-convolution weights: K reordered to (dy, dx, within-block) -- see riqn_conv_fwd_strip
        if getattr(self, "_strip_ops", None) is None or self._strip_ops["conv1"][0].device != dev:
            self._strip_perm = {n: _strip_perm(cin, k, st, first).to(dev) for n, cin, k, st, first in
                                (("conv1", self.history, 8, 4, True), ("conv2", 32, 4, 2, False), ("conv3", 64, 3, 1, False))}
            self._strip_perm32 = {n: pm.to(torch.int32) for n, pm in self._strip_perm.items()}
            self._strip_ops = {n: (torch.empty(co, pm.numel(), dtype=torch.bfloat16, device=dev),
                                   torch.empty(co, pm.numel(), dtype=torch.bfloat16, device=dev))
                               for (n, pm), co in zip(self._strip_perm.items(), (32, 64, 64))}
            self._split_jobs = None
        # every noise-free weight image in ONE launch (riqn_split_bf16_multi); the job table only holds static addresses
        convs = (("conv1", self.conv1), ("conv2", self.conv2), ("conv3", self.conv3))
        key = tuple(c.weight.data_ptr() for _, c in convs) + (self._strip_ops["conv1"][0].data_ptr(),)
        if getattr(self, "_split_jobs", None) is None or self._split_jobs[0] != key:
            specs = []
            for name, conv in convs:
                hi, lo, hiT = self._conv_ops[name]
                specs.append((conv.weight, None, 1.0, hi, lo, hiT))                       # original k order (+ transpose)
                shi, slo = self._strip_ops[name]
                specs.append((conv.weight, self._strip_perm32[name], 255.0 if name == "conv1" else 1.0, shi, slo, None))
            specs.append((self.conv1.weight, None, 255.0, self._conv1_px_ops[0], self._conv1_px_ops[1], None))
            if not self.rainbow_only:
                specs.append((self.iqn_fc.weight, None, 1.0, self._iqn_ops[0], self._iqn_ops[1], None))
            arr = (SplitJob * len(specs))()
            for j, (src, perm, div, hi, lo, hiT) in zip(arr, specs):
                j.src, j.perm = src.data_ptr(), perm.data_ptr() if perm is not None else None
                j.rows, j.cols, j.div = hi.shape[0], hi.shape[1], div
                j.hi, j.lo, j.hi_t = hi.data_ptr(), lo.data_ptr(), hiT.data_ptr() if hiT is not None else None
            self._split_jobs = (key, arr, len(specs))
        call("riqn_split_bf16_multi", self._split_jobs[2], self._split_jobs[1])

    def _support(self, dev):
        """z-support of the categorical head (agent.py:54-57); only used when forward() is called without an Agent."""
        if getattr(self, "_support_t", None) is None or self._support_t.device != dev:
            self._support_t = torch.linspace(self._v_min, self._v_max, self.atoms).to(dev)
        return self._support_t

    def begin_step(self, dyn=None):
        """Reset the per-step Philox stream indices (CUDA-graph mode keeps them static across replays)."""
        self._dyn = dyn
        self._tau_in_step = 0
        for _, m in self.noisy_layers():
            m._dyn = dyn
            m._calls_in_step = 0

    def draw_quantiles(self, n):
        tau = torch.empty(n, 1, device=self._flat.device)
        dyn = getattr(self, "_dyn", None)
        idx = self._tau_in_step if dyn is not None else self._tau_calls
        call("riqn_fill_uniform", n, self._rng_seed ^ 0x7A75, self._tau_stream_offset + idx + (0 if dyn is not None else _EAGER_STREAMS), ptr(tau),
             dyn.ptr() if dyn else None)
        self._tau_calls += 1
        self._tau_in_step += 1
        return tau

    # ------------------------------------------------------------------ forward pieces
    def trunk(self, x, keep=None, col_cache=None):
        """conv1-3 + ReLU -> (B, 3136).  x: (B, history, 84, 84) uint8 (scaled by 1/255 on the fly) or
        fp32; may be a view with a larger batch stride (the replay window).  model.py:115-118"""
        _lib.require_device()
        B = x.shape[0]
        if x.dtype not in (torch.uint8, torch.float32):
            x = x.float()
        if x.stride()[1:] != (84 * 84, 84, 1):
            x = x.contiguous()
        is_u8 = 1 if x.dtype == torch.uint8 else 0
        dev = x.device
        g1 = _geom(B, self.history, 84, 32, 8, 4, 1, in_bstride=x.stride(0))
        g2 = _geom(B, 32, 20, 64, 4, 2, 0)
        g3 = _geom(B, 64, 9, 64, 3, 1, 0)
        geoms, convs = (g1, g2, g3), (self.conv1, self.conv2, self.conv3)
        outs = (torch.empty(B, 32, 20, 20, device=dev), torch.empty(B, 64, 9, 9, device=dev),
                torch.empty(B, 64, 7, 7, device=dev))
        ins = (x, outs[0], outs[1])
        fwd = PRECISION["fwd"]
        # the backward runs on the tensor cores when it is bf16 and every im2col row count is a multiple of 8
        bwd_tc = keep is not None and PRECISION["bwd"] == "bf16" and fwd != "fp32" and all((g.B * g.OH * g.OW) % 8 == 0 for g in geoms)
        need_col32 = keep is not None and not bwd_tc
        cols, colTs = [None] * 3, [None] * 3
        px_scale = 1.0
        strip = (fwd != "fp32" and is_u8 and x.stride(0) % 16 == 0 and x.data_ptr() % 16 == 0 and self.history * 16 == 64
                 and not _NO_STRIP)
        if strip:
            # strip convolution (riqn_conv_fwd_strip): no im2col matrices in the forward; each layer's epilogue writes
            # the next layer's block matrix.  Block grids: G = OH + k/stride - 1 = 21, 10, 9.
            x3 = _small_x3()
            bf = lambda *sh: torch.empty(*sh, dtype=torch.bfloat16, device=dev)
            ckey = ("s2d", x.data_ptr(), tuple(x.shape), tuple(x.stride()))
            if col_cache is not None and ckey in col_cache:
                a1 = col_cache[ckey]                 # the pixel block matrix does not depend on the network's weights
            else:
                a1 = bf(B * 21 * 21, 16 * self.history)
                call("riqn_s2d_u8", g1, ptr(x), ptr(a1))
                if col_cache is not None:
                    col_cache[ckey] = a1
            a2_hi, a2_lo = bf(B * 100, 128), (bf(B * 100, 128) if x3 else None)
            a3_hi, a3_lo = bf(B * 81, 64), (bf(B * 81, 64) if x3 else None)
            ops = self._strip_ops
            # the fp32 NCHW activations of conv1 / conv2 are only read by the backward (ReLU masks): no-grad passes skip them
            o1, o2 = (ptr(outs[0]), ptr(outs[1])) if keep is not None else (None, None)
            call("riqn_conv_fwd_strip", g1, ptr(a1), None, ptr(ops["conv1"][0]), ptr(ops["conv1"][1]) if x3 else None,
                 ptr(self.conv1.bias), o1, ptr(a2_hi), ptr(a2_lo), 2, 10, None, None, None, 0)
            call("riqn_conv_fwd_strip", g2, ptr(a2_hi), ptr(a2_lo), ptr(ops["conv2"][0]), ptr(ops["conv2"][1]) if x3 else None,
                 ptr(self.conv2.bias), o2, ptr(a3_hi), ptr(a3_lo), 1, 9, None, None, None, 0)
            call("riqn_conv_fwd_strip", g3, ptr(a3_hi), ptr(a3_lo), ptr(ops["conv3"][0]), ptr(ops["conv3"][1]) if x3 else None,
                 ptr(self.conv3.bias), ptr(outs[2]), None, None, 0, 0, None, None, None, 0)
            if keep is not None:                     # operands of the backward products
                strip_bwd = None
                if bwd_tc:                           # the strip backward reads the forward's block matrices
                    strip_bwd = (a1, a2_hi, a3_hi)
                    px_scale = 1.0 / 255.0
                else:
                    for i, (g, inp) in enumerate(zip(geoms, ins)):
                        M, K = g.B * g.OH * g.OW, g.Cin * g.KH * g.KW
                        cols[i] = torch.empty(M, K, device=dev)
                        call("riqn_im2col_f32", g, ptr(inp), 1 if i == 0 else 0, ptr(cols[i]))
                keep.update(x=x, g=geoms, col=tuple(cols), colT=tuple(colTs), out=outs, bwd_tc=bwd_tc, px_scale=px_scale,
                            strip_bwd=strip_bwd)
            return outs[2].view(B, FEAT)
        for i, (g, conv, inp, out) in enumerate(zip(geoms, convs, ins, outs)):
            M, K = g.B * g.OH * g.OW, g.Cin * g.KH * g.KW
            u8 = is_u8 if i == 0 else 0
            if fwd == "fp32":
                cols[i] = torch.empty(M, K, device=dev)
                call("riqn_conv_fwd", g, ptr(inp), u8, ptr(conv.weight), ptr(conv.bias), ptr(cols[i]), ptr(out))
            elif i == 0 and u8 and x.stride(0) % 16 == 0 and x.data_ptr() % 16 == 0:
                # raw-pixel path: pixel values are exact in bf16, /255 folded into the weights
                ws_hi, ws_lo = self._conv1_px_ops
                ckey = (x.data_ptr(), tuple(x.shape), tuple(x.stride()))
                reuse = col_cache is not None and ckey in col_cache and not bwd_tc
                col_px = col_cache[ckey] if reuse else torch.empty(M, K, dtype=torch.bfloat16, device=dev)
                if col_cache is not None:
                    col_cache[ckey] = col_px          # the pixel im2col does not depend on the network's weights
                if bwd_tc:
                    colTs[i] = torch.empty(K, M, dtype=torch.bfloat16, device=dev)
                    px_scale = 1.0 / 255.0
                call("riqn_conv_fwd_tc_u8", g, ptr(inp), ptr(ws_hi), ptr(ws_lo) if _small_x3() else None, ptr(conv.bias),
                     ptr(col_px), ptr(colTs[i]), ptr(out), 1 if reuse else 0)
                if need_col32:
                    cols[i] = torch.empty(M, K, device=dev)
                    call("riqn_im2col_f32", g, ptr(inp), u8, ptr(cols[i]))
            else:
                w_hi, w_lo, _ = self._conv_ops["conv%d" % (i + 1)]
                col_hi = torch.empty(M, K, dtype=torch.bfloat16, device=dev)
                col_lo = torch.empty(M, K, dtype=torch.bfloat16, device=dev) if _small_x3() else None
                if bwd_tc:
                    colTs[i] = torch.empty(K, M, dtype=torch.bfloat16, device=dev)
                call("riqn_conv_fwd_tc", g, ptr(inp), u8, ptr(w_hi), ptr(w_lo), ptr(conv.bias), ptr(col_hi), ptr(col_lo),
                     ptr(colTs[i]), ptr(out))
                if need_col32:
                    cols[i] = torch.empty(M, K, device=dev)
                    call("riqn_im2col_f32", g, ptr(inp), u8, ptr(cols[i]))
        if keep is not None:
            keep.update(x=x, g=geoms, col=tuple(cols), colT=tuple(colTs), out=outs, bwd_tc=bwd_tc, px_scale=px_scale)
        return outs[2].view(B, FEAT)

    def trunk_pair(self, other, x):
        """conv1-3 of TWO networks (self = online, other = target) over the same uint8 frames in three launches instead of
        six (no-grad passes: compute_loss_iqn.py:235,256 both read next_states).  The batch is stacked -- samples [0, B) with
        self's weights, [B, 2B) with other's -- the pixel block matrix is shared by both halves.  Returns (feat_self,
        feat_other), each (B, 3136); None when the fast path does not apply (the caller then runs the trunks one by one)."""
        B = x.shape[0]
        if (PRECISION["fwd"] == "fp32" or _NO_STRIP or x.dtype != torch.uint8 or x.stride()[1:] != (84 * 84, 84, 1)
                or x.stride(0) % 16 or x.data_ptr() % 16 or self.history != 4 or other.history != 4 or B % 128):
            return None
        for net in (self, other):                      # operand images of the noise-free weights (rebuilt only when dirty)
            if getattr(net, "_strip_ops", None) is None or getattr(net, "_static_ops_dirty", True):
                net._refresh_tc_operands(h_done=True)
        dev = x.device
        x3 = _small_x3()
        bf = lambda *sh: torch.empty(*sh, dtype=torch.bfloat16, device=dev)
        g1 = _geom(B, self.history, 84, 32, 8, 4, 1, in_bstride=x.stride(0))
        a1 = bf(B * 21 * 21, 16 * self.history)
        call("riqn_s2d_u8", g1, ptr(x), ptr(a1))
        g1p, g2p, g3p = _geom(2 * B, self.history, 84, 32, 8, 4, 1), _geom(2 * B, 32, 20, 64, 4, 2, 0), _geom(2 * B, 64, 9, 64, 3, 1, 0)
        a2_hi, a2_lo = bf(2 * B * 100, 128), (bf(2 * B * 100, 128) if x3 else None)
        a3_hi, a3_lo = bf(2 * B * 81, 64), (bf(2 * B * 81, 64) if x3 else None)
        feat = torch.empty(2 * B, FEAT, device=dev)
        so, oo = self._strip_ops, other._strip_ops
        lo = lambda t: ptr(t) if x3 else None
        call("riqn_conv_fwd_strip", g1p, ptr(a1), None, ptr(so["conv1"][0]), lo(so["conv1"][1]), ptr(self.conv1.bias), None,
             ptr(a2_hi), ptr(a2_lo), 2, 10, ptr(oo["conv1"][0]), lo(oo["conv1"][1]), ptr(other.conv1.bias), 1)
        call("riqn_conv_fwd_strip", g2p, ptr(a2_hi), ptr(a2_lo), ptr(so["conv2"][0]), lo(so["conv2"][1]), ptr(self.conv2.bias), None,
             ptr(a3_hi), ptr(a3_lo), 1, 9, ptr(oo["conv2"][0]), lo(oo["conv2"][1]), ptr(other.conv2.bias), 0)
        call("riqn_conv_fwd_strip", g3p, ptr(a3_hi), ptr(a3_lo), ptr(so["conv3"][0]), lo(so["conv3"][1]), ptr(self.conv3.bias),
             ptr(feat), None, None, 0, 0, ptr(oo["conv3"][0]), lo(oo["conv3"][1]), ptr(other.conv3.bias), 0)
        return feat[:B], feat[B:]

    def iqn_head(self, feat, num_quantiles, tau, keep=None):
        """Quantile embedding, Hadamard, noisy hidden layers, z-layers, dueling.  model.py:131-157"""
        B = feat.shape[0]
        R = B * num_quantiles
        dev = feat.device
        E, hid, A = self.quantile_embedding_dim, self.hidden, self.action_space
        fwd, bwd = PRECISION["fwd"], PRECISION["bwd"]
        bf = lambda *sh: torch.empty(*sh, dtype=torch.bfloat16, device=dev)
        h = torch.empty(R, 2 * hid, device=dev)
        bwd_tc = keep is not None and bwd != "fp32" and R % 8 == 0      # head wgrad/dgrad on the tensor cores
        emb_tc = keep is not None and bwd == "bf16" and fwd != "fp32" and R % 8 == 0   # embedding backward on tensor cores
        cosv = xt = tc = None
        if fwd == "fp32":
            cosv = torch.empty(R, E, device=dev)
            xt = torch.empty(R, FEAT, device=dev)
            call("riqn_quantile_embed_fwd", B, num_quantiles, E, FEAT, ptr(tau), ptr(feat), ptr(self.iqn_fc.weight),
                 ptr(self.iqn_fc.bias), ptr(cosv), ptr(xt))
            if bwd_tc:
                tc = dict(x_hi=None, x_lo=None, x_hiT=bf(FEAT, R), x_loT=bf(FEAT, R) if bwd == "bf16x3" else None)
                call("riqn_split_bf16", R, FEAT, ptr(xt), None, None, ptr(tc["x_hiT"]), ptr(tc["x_loT"]), 0)
            call("riqn_noisy_linear_fwd", R, FEAT, 2 * hid, ptr(xt), ptr(self._w_eff_h), ptr(self._b_eff_h), ptr(h))
        else:
            x3 = _small_x3()                                     # embedding product
            f16 = fwd == "fp16"                                  # head product: one pass on fp16 images
            head_x3 = fwd == "bf16x3"
            need_x32 = keep is not None and not emb_tc           # the fp32 CUDA-core embedding backward reads x
            # bwd == "bf16": the weight-gradient products read the row-major images (MN-major operands): no transposes
            mn = bwd_tc and bwd == "bf16"
            # fp16 mode: x_hi = fp16(x) feeds the forward product; the gradient pass also keeps x_bf = bf16(x) (written into
            # the lo slot by the same epilogue) for the weight-gradient product and the embedding backward
            tc = dict(x_hi=torch.empty(R, FEAT, dtype=torch.float16 if f16 else torch.bfloat16, device=dev),
                      x_lo=bf(R, FEAT) if (head_x3 or (f16 and keep is not None)) else None, f16=f16,
                      x_hiT=bf(FEAT, R) if (bwd_tc and not mn) else None,
                      x_loT=bf(FEAT, R) if (bwd_tc and bwd == "bf16x3") else None,
                      cos_hi=bf(R, E), cos_lo=bf(R, E) if x3 else None, cosT_hi=None, mn=mn)
            if need_x32:
                xt = torch.empty(R, FEAT, device=dev)
                cosv = torch.empty(R, E, device=dev)
            elif tc["x_hiT"] is not None:                        # transposed images are split from the fp32 matrix
                xt = torch.empty(R, FEAT, device=dev)
            call("riqn_quantile_embed_fwd_tc", B, num_quantiles, E, FEAT, ptr(tau), ptr(feat), ptr(self._iqn_ops[0]),
                 ptr(self._iqn_ops[1]), ptr(self.iqn_fc.bias), ptr(tc["cos_hi"]), ptr(tc["cos_lo"]), ptr(tc["cosT_hi"]),
                 ptr(xt), ptr(tc["x_hi"]), ptr(tc["x_lo"]), ptr(tc["x_hiT"]), ptr(tc["x_loT"]), 1 if f16 else 0)
            if need_x32:   # fp32 cos for the CUDA-core dW_e product
                call("riqn_quantile_embed_fwd", B, num_quantiles, E, FEAT, ptr(tau), ptr(feat), ptr(self.iqn_fc.weight),
                     ptr(self.iqn_fc.bias), ptr(cosv), ptr(xt))
            tc["h_hi"] = bf(R, 2 * hid) if (bwd_tc and R % 2 == 0) else None   # bf16 image of h for the z-layer weight gradient
            call("riqn_gemm_bf16_tc", R, 2 * hid, FEAT, ptr(tc["x_hi"]), ptr(tc["x_lo"]) if head_x3 else None, ptr(self._w_hi),
                 ptr(self._w_lo) if head_x3 else None, ptr(h), 2 * hid, 1, ptr(self._b_eff_h), None, None, 1, None, ptr(tc["h_hi"]),
                 3 if f16 else 0)
        q = torch.empty(R, A, device=dev)
        call("riqn_dueling_fwd", R, B, hid, A, ptr(h), ptr(self._w_eff_z), ptr(self._b_eff_z), ptr(q))
        if keep is not None:
            keep.update(feat=feat, cos=cosv, xt=xt, h=h, q=q, tau=tau, num_quantiles=num_quantiles, tc=tc,
                        noise_version=getattr(self, "_noise_version", 0),
                        head_bwd_tc=bwd_tc, emb_bwd_tc=emb_tc)
        return q

    def forward(self, x, num_quantiles=None, log=False, tau=None, keep=None, fresh_weights=False, col_cache=None, feat=None):
        """model.py:112-157.  Returns (q, quantiles) in IQN mode.  ``feat`` (B, 3136): trunk output computed by the caller
        (trunk_pair); only valid for no-grad passes."""
        if self.rainbow_only:
            from . import c51
            return c51.forward(self, x, log=log, keep=keep, fresh_weights=fresh_weights)
        if not fresh_weights:
            self.compose_weights()
        if feat is None or keep is not None:
            feat = self.trunk(x, keep, col_cache)
        if tau is None:
            tau = self.draw_quantiles(num_quantiles * x.shape[0])
        else:
            tau = tau.to(feat.device, torch.float32).reshape(-1, 1).contiguous()
        q = self.iqn_head(feat, num_quantiles, tau, keep)
        return q, tau

    # ------------------------------------------------------------------ backward of forward()
    def backward_iqn(self, keep, dtheta, gscale, actions, gscale_mul=1.0):
        """Accumulate dL/dparams into the gradient arena for the forward recorded in ``keep``, where
        dL/dq[r, actions[b]] = dtheta[r] * gscale[b] * gscale_mul  (r = quantile*B + b)."""
        if keep.get("noise_version", None) != getattr(self, "_noise_version", 0):
            raise RuntimeError("the network's noise was resampled between this forward pass and its backward: the composed "
                               "weights / epsilons of the gradient pass are gone (call backward before the next reset_noise)")
        B = keep["feat"].shape[0]
        Nq = keep["num_quantiles"]
        R = B * Nq
        dev = keep["feat"].device
        hid, A, E = self.hidden, self.action_space, self.quantile_embedding_dim
        hv, ha, zv, za = self.fcnoisy_h_v, self.fcnoisy_h_a, self.fcnoisy_z_v, self.fcnoisy_z_a
        gv = self.grad_view
        dz = torch.empty(R, 32, device=dev)
        tc = keep.get("tc")
        f16 = bool(tc and tc.get("f16"))
        x_bf = tc["x_lo"] if f16 else (tc["x_hi"] if tc else None)      # bf16 image of x (fp16 forward: the second image)
        w_bf = self._w_lo if f16 else getattr(self, "_w_hi", None)      # bf16 image of W_eff
        z_tc = bool(keep["head_bwd_tc"]) and tc is not None and tc.get("h_hi") is not None
        dzT = torch.empty(R, 32, dtype=torch.bfloat16, device=dev) if z_tc else None       # (R, 32) row-major bf16 image
        dbs = torch.empty(2 * hid, device=dev)
        # bf16 backward: dh leaves the dueling backward directly as the bf16 operand images (+ its column sums)
        fused_dh = bool(keep["head_bwd_tc"]) and PRECISION["bwd"] == "bf16" and R % 8 == 0 and bool(tc and tc.get("mn"))
        if fused_dh:
            dh = None
            dh_hi = torch.empty(R, 2 * hid, dtype=torch.bfloat16, device=dev)
            dh_hiT = None                            # the wgrad reads dh_hi itself (MN-major operand)
            call("riqn_dueling_bwd_bf16", R, B, hid, A, ptr(keep["h"]), ptr(tc.get("h_hi")), ptr(self._w_eff_z), ptr(dtheta), ptr(gscale),
                 float(gscale_mul), ptr(actions), ptr(dh_hi), None, ptr(dbs), ptr(dz), ptr(dzT))
        else:
            dh = torch.empty(R, 2 * hid, device=dev)
            call("riqn_dueling_bwd", R, B, hid, A, ptr(keep["h"]), ptr(self._w_eff_z), ptr(dtheta), ptr(gscale),
                 float(gscale_mul), ptr(actions), ptr(dh), ptr(dz), ptr(dzT))
        dwz = torch.empty(32, 2 * hid, device=dev)
        dbz = torch.empty(32, device=dev)
        zargs = (ptr(dwz), ptr(dbz), ptr(zv.weight_epsilon), ptr(zv.bias_epsilon), ptr(za.weight_epsilon),
                 ptr(za.bias_epsilon), ptr(gv(zv.weight_mu)), ptr(gv(zv.weight_sigma)), ptr(gv(zv.bias_mu)),
                 ptr(gv(zv.bias_sigma)), ptr(gv(za.weight_mu)), ptr(gv(za.weight_sigma)), ptr(gv(za.bias_mu)),
                 ptr(gv(za.bias_sigma)))
        if z_tc:
            call("riqn_z_wgrad_tc", R, hid, A, ptr(dzT), ptr(tc["h_hi"]), ptr(dz), *zargs)
        else:
            call("riqn_z_wgrad", R, hid, A, ptr(dz), ptr(keep["h"]), *zargs)
        bwd = PRECISION["bwd"]
        # bf16 backward: dx is consumed as a bf16 operand anyway, so the dgrad writes it as bf16 (half the traffic)
        dx_bf16 = fused_dh and bool(keep["emb_bwd_tc"])
        dx = torch.empty(R, FEAT, dtype=torch.bfloat16 if dx_bf16 else torch.float32, device=dev)
        # [h_v | h_a] are adjacent in every arena, so one (2*hid, 3136) product serves both layers
        if not keep["head_bwd_tc"]:
            call("riqn_noisy_linear_wgrad", R, FEAT, 2 * hid, ptr(dh), ptr(keep["xt"]), ptr(hv.weight_epsilon),
                 ptr(hv.bias_epsilon), ptr(dbs), ptr(gv(hv.weight_mu)), ptr(gv(hv.weight_sigma)), ptr(gv(hv.bias_mu)),
                 ptr(gv(hv.bias_sigma)))
            call("riqn_noisy_linear_dgrad", R, FEAT, 2 * hid, ptr(dh), ptr(self._w_eff_h), ptr(dx))
        else:
            bf = lambda *sh: torch.empty(*sh, dtype=torch.bfloat16, device=dev)
            b3 = bwd == "bf16x3"
            dh_lo, dh_loT = (bf(R, 2 * hid), bf(2 * hid, R)) if b3 else (None, None)
            if not fused_dh:
                dh_hi, dh_hiT = bf(R, 2 * hid), bf(2 * hid, R)
                call("riqn_split_bf16", R, 2 * hid, ptr(dh), ptr(dh_hi), ptr(dh_lo), ptr(dh_hiT), ptr(dh_loT), 0)
            # dW[o, i] = sum_r dh[r, o] x[r, i]  -> dmu += dW, dsigma += dW * eps   (split-K, atomics)
            if fused_dh:
                call("riqn_gemm_bf16_tc_mn", 2 * hid, FEAT, R, ptr(dh_hi), ptr(x_bf), 1, ptr(gv(hv.weight_mu)), FEAT, 3,
                     ptr(gv(hv.weight_sigma)), ptr(hv.weight_epsilon), 1.0, WGRAD_SPLIT_K, None, 0)
            else:
                call("riqn_gemm_bf16_tc", 2 * hid, FEAT, R, ptr(dh_hiT), ptr(dh_loT), ptr(tc["x_hiT"]),
                     ptr(tc["x_loT"]) if b3 else None, ptr(gv(hv.weight_mu)), FEAT, 3, None, ptr(gv(hv.weight_sigma)),
                     ptr(hv.weight_epsilon), WGRAD_SPLIT_K, None, None, 0)
            call("riqn_noisy_bias_grad", R, 2 * hid, ptr(dh) if dh is not None else None, ptr(hv.bias_epsilon), ptr(dbs),
                 ptr(gv(hv.bias_mu)), ptr(gv(hv.bias_sigma)))
            # from here on the gradients of every NoisyLinear layer (the arena from fcnoisy_h_v.weight_mu to its end, 96% of
            # the bytes) are final: a data-parallel learner starts their all-reduce now, under the rest of the backward
            hook = getattr(self, "_grads_ready_hook", None)
            if hook is not None:
                hook(self._offsets[id(hv.weight_mu)])
            # dx[r, i] = sum_o dh[r, o] W_eff[o, i]
            if fused_dh:     # W_eff (2*hid, 3136) itself is the (K, N) operand: no transposed weight image
                call("riqn_gemm_bf16_tc_mn", R, FEAT, 2 * hid, ptr(dh_hi), ptr(w_bf), 0, None if dx_bf16 else ptr(dx), FEAT,
                     0, None, None, 1.0, 1, ptr(dx) if dx_bf16 else None, 0)
            else:
                call("riqn_gemm_bf16_tc", R, FEAT, 2 * hid, ptr(dh_hi), ptr(dh_lo), ptr(self._w_hiT),
                     ptr(self._w_loT) if b3 else None, ptr(dx), FEAT, 0, None, None, None, 1, None, None, 0)
        dfeat = torch.empty(B, FEAT, device=dev)
        if keep["emb_bwd_tc"]:
            dpre = torch.empty(R, FEAT, dtype=torch.bfloat16, device=dev)
            # bf16 backward: x = x_hi (the lo image only refines the forward)
            call("riqn_quantile_embed_bwd_tc", B, Nq, E, FEAT, ptr(x_bf), None if (dx_bf16 or f16) else ptr(tc["x_lo"]),
                 ptr(keep["feat"]), ptr(tc["cos_hi"]), ptr(dx), 1 if dx_bf16 else 0, ptr(dpre), ptr(dfeat),
                 ptr(gv(self.iqn_fc.weight)), ptr(gv(self.iqn_fc.bias)))
        else:
            call("riqn_quantile_embed_bwd", B, Nq, E, FEAT, ptr(keep["xt"]), ptr(keep["feat"]), ptr(keep["cos"]), ptr(dx),
                 ptr(dfeat), ptr(gv(self.iqn_fc.weight)), ptr(gv(self.iqn_fc.bias)))
        self.backward_trunk(keep, dfeat)

    def backward_trunk(self, keep, dfeat):
        (g1, g2, g3), (out1, out2, out3) = keep["g"], keep["out"]
        dev = dfeat.device
        gv = self.grad_view
        convs = (self.conv1, self.conv2, self.conv3)
        douts = [None, None, dfeat]
        for i in (2, 1, 0):
            g, conv, out = keep["g"][i], convs[i], keep["out"][i]
            M, K = g.B * g.OH * g.OW, g.Cin * g.KH * g.KW
            din = torch.empty_like(keep["out"][i - 1]) if i > 0 else None
            if keep["bwd_tc"] and keep.get("strip_bwd") is not None:
                name = "conv%d" % (i + 1)
                w_hi = self._conv_ops[name][0]                 # (Cout, K) in the original k order
                G = g.OH + g.KH // g.stride - 1
                dYg = torch.empty(g.B * G * G, g.Cout, dtype=torch.bfloat16, device=dev)
                dwp = torch.empty(g.Cout, K, device=dev)
                call("riqn_conv_bwd_strip", g, ptr(douts[i]), ptr(out), ptr(keep["strip_bwd"][i]), ptr(w_hi),
                     ptr(self._strip_perm32[name]), ptr(dYg), ptr(dwp), ptr(gv(conv.weight)), ptr(gv(conv.bias)), ptr(din),
                     keep["px_scale"] if i == 0 else 1.0)
            elif keep["bwd_tc"]:
                _, _, wT_hi = self._conv_ops["conv%d" % (i + 1)]
                dY = torch.empty(M, g.Cout, dtype=torch.bfloat16, device=dev) if i > 0 else None
                dYT = torch.empty(g.Cout, M, dtype=torch.bfloat16, device=dev)
                dcol = torch.empty(M, K, device=dev) if i > 0 else None
                call("riqn_conv_bwd_tc", g, ptr(douts[i]), ptr(out), ptr(keep["colT"][i]), ptr(wT_hi), ptr(dY), ptr(dYT),
                     ptr(dcol), ptr(gv(conv.weight)), ptr(gv(conv.bias)), ptr(din), keep["px_scale"] if i == 0 else 1.0)
            else:
                dY = torch.empty(M, g.Cout, device=dev)
                dcol = torch.empty(M, K, device=dev) if i > 0 else None
                call("riqn_conv_bwd", g, ptr(douts[i]), ptr(out), ptr(keep["col"][i]), ptr(conv.weight), ptr(dY), ptr(dcol),
                     ptr(gv(conv.weight)), ptr(gv(conv.bias)), ptr(din))
            if i > 0:
                douts[i - 1] = din
