"""GPU: the data gradient of riqn_conv_bwd_strip (the shifted-row gather product, TC_DGRAD in csrc/gemm_tc.cu) against a
float64 product of the same bf16 operands -- the dYg the call wrote and the bf16 weight -- so that only the fp32
accumulation order differs; every din element is written exactly once and the result is run-to-run identical."""
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu

# (Cin, H, Cout, k, stride): conv2 and conv3 of the DQN trunk, and a conv2-like layer whose image has a remainder row /
# column that no output reads (H - k not a multiple of the stride)
LAYERS = {"conv2": (32, 20, 64, 4, 2), "conv3": (64, 9, 64, 3, 1), "conv2_remainder": (32, 21, 64, 4, 2)}


def _setup(dev, name, batch, seed):
    import torch.nn.functional as F
    from rainbow_iqn_apex_b200._lib import ConvGeom
    from rainbow_iqn_apex_b200.model import _strip_perm
    cin, h, cout, k, s = LAYERS[name]
    oh = (h - k) // s + 1
    G = oh + k // s - 1
    K = cin * k * k
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(cout, K, generator=g) / K ** 0.5
    ins = dict(
        geom=ConvGeom(batch, cin, h, h, cout, k, k, s, 0, oh, oh, cin * h * h),
        dout=torch.randn(batch, cout, oh, oh, generator=g).to(dev),
        out=torch.randn(batch, cout, oh, oh, generator=g).to(dev),          # ~half the ReLU mask open
        a_hi=torch.randn(batch * G * G, s * s * cin, generator=g).to(torch.bfloat16).to(dev),
        w_hi=w.to(torch.bfloat16).to(dev),
        perm=_strip_perm(cin, k, s, False).to(torch.int32).to(dev),
        dYg=torch.empty(batch * G * G, cout, dtype=torch.bfloat16, device=dev),
        dwp=torch.empty(cout, K, device=dev),
        dw=torch.zeros(cout, K, device=dev),
        db=torch.zeros(cout, device=dev),
    )
    return ins, (cin, h, cout, k, s, oh, G, F)


def _call(ins, din):
    from rainbow_iqn_apex_b200._lib import call, ptr
    call("riqn_conv_bwd_strip", ins["geom"], ptr(ins["dout"]), ptr(ins["out"]), ptr(ins["a_hi"]), ptr(ins["w_hi"]),
         ptr(ins["perm"]), ptr(ins["dYg"]), ptr(ins["dwp"]), ptr(ins["dw"]), ptr(ins["db"]), ptr(din), 1.0)
    torch.cuda.synchronize()


@pytest.mark.parametrize("batch", [3, 8, 512])
@pytest.mark.parametrize("name", sorted(LAYERS))
def test_strip_dgrad_matches_float64_product(cuda_dev, name, batch):
    """din against conv_transpose2d in float64 of the call's own bf16 dYg and the bf16 weight (bound 1e-5 relative).
    din starts as NaN: every element must come back written (the remainder row / column as zeros)."""
    ins, (cin, h, cout, k, s, oh, G, F) = _setup(cuda_dev, name, batch, seed=100 + batch)
    din = torch.full((batch, cin, h, h), float("nan"), device=cuda_dev)
    _call(ins, din)
    assert not torch.isnan(din).any()
    dyg = ins["dYg"].double().view(batch, G, G, cout)
    assert not dyg[:, oh:].any() and not dyg[:, :, oh:].any()        # the grid's padding rows are zeros
    dy = dyg[:, :oh, :oh].permute(0, 3, 1, 2)
    ref = F.conv_transpose2d(dy, ins["w_hi"].double().view(cout, cin, k, k), stride=s)
    full = torch.zeros(batch, cin, h, h, dtype=torch.float64, device=cuda_dev)
    full[:, :, :ref.shape[2], :ref.shape[3]] = ref
    err = rel_err(din.cpu().numpy(), full.cpu().numpy())
    assert err < 1e-5, err


@pytest.mark.parametrize("name", ["conv2", "conv3"])
def test_strip_dgrad_bitwise_repeatable(cuda_dev, name):
    """Two calls on the same inputs give bit-identical din (plain stores in a fixed accumulation order)."""
    ins, (cin, h, *_rest) = _setup(cuda_dev, name, 512, seed=7)
    d1 = torch.empty(512, cin, h, h, device=cuda_dev)
    d2 = torch.full_like(d1, float("nan"))
    _call(ins, d1)
    _call(ins, d2)
    assert torch.equal(d1, d2)
