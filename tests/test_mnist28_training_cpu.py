"""CPU: the training step's orchestration on the MNIST-style 28x28 geometry (BASELINE configs[3]: 1 channel, 28 -> 14 -> 7), and
wgrad's one remaining size refusal.

The graph runs on the fp64 contract model of the kernels (ContractOps, tests/test_training_graph.py) and is compared with autograd
through the oracle UNet.  Sizes that are not powers of two reach every place the graph could assume one: the 14 <-> 28 and 7 <-> 14
resample adjoints, attention at N = 784 / 196 / 49, and in_conv's im2col GEMM with 9 real patch columns of 128.
"""
import ctypes as C
import math
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import make_state_dict                                       # noqa: E402
from oracle.unet_ref import _unet_forward                                # noqa: E402
from tests.cases import UNET_CASES                                       # noqa: E402
from tests.test_training_graph import ContractOps                        # noqa: E402
from v_diffusion_b200 import UNet, _lib                                  # noqa: E402
from v_diffusion_b200.training import UNetTrainGraph                     # noqa: E402


@pytest.fixture
def mnist_contract_ops(monkeypatch):
    import v_diffusion_b200.training as T
    ops = ContractOps()
    monkeypatch.setattr(T, "KernelOps", lambda operand_dtype="fp16": ops)
    return ops


def test_mnist28_graph_orchestration_matches_autograd(mnist_contract_ops):
    """Output and every parameter gradient of UNetTrainGraph on UNET_CASES["mnist28"] at 28x28, B = 3 with an unconditional
    row, against fp32 autograd through the oracle UNet; the bars of test_graph_orchestration_matches_autograd."""
    cfg, B, R = UNET_CASES["mnist28"]["cfg"], 3, 28
    sd = make_state_dict(cfg, 5)
    net = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"], cfg["num_res_blocks"],
               cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], head_dim=cfg["head_dim"], num_heads=cfg["num_heads"],
               num_classes=cfg["num_classes"], multitags=cfg["multitags"])
    net.load_state_dict(sd, strict=True)
    net = net.double()
    g = torch.Generator().manual_seed(28)
    x = torch.randn(B, 1, R, R, generator=g)
    t = torch.rand(B, generator=g, dtype=torch.float64)
    go = torch.randn(B, 1, R, R, generator=g)
    y = torch.tensor([4, 0, 10])                                           # label 0: the unconditional row

    graph = UNetTrainGraph(net)
    out = graph.forward(x.double(), t, y)
    grads = graph.backward(go.double())
    ref_sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    with torch.enable_grad():
        ref = _unet_forward(ref_sd, cfg, x, t, y, None)
        ref.backward(go)

    assert out.shape == ref.shape == (B, 1, R, R)
    out_rel = ((out - ref.detach().double()).norm() / ref.detach().double().norm()).item()
    assert out_rel < 2e-5, out_rel
    assert set(grads) == set(sd) and len(sd) == 236
    worst = {}
    for k in sd:
        want = ref_sd[k].grad.double()
        assert grads[k].shape == want.shape, k
        worst[k] = (grads[k].double() - want).norm().item() / (want.norm().item() + 2e-5 * math.sqrt(want.numel()))
    bad = {k: v for k, v in worst.items() if v > 2e-4}
    assert not bad, bad
    for fam in ("conv1", "conv3", "attention", "conv_backward1", "conv_backward3", "groupnorm_backward", "attention_backward"):
        assert fam in mnist_contract_ops.calls, fam


def test_wgrad_still_refuses_maps_wider_than_128():
    """Any feature map the forward conv takes now trains; a 130-wide one is refused with conv_geom's message before any
    device call."""
    L = _lib.lib()
    dummy = C.c_void_p(0x1000)                                             # never dereferenced: the size check fires first
    rc = L.vdt_op_conv_wgrad(dummy, dummy, 1, 4, 130, 64, 64, 3, dummy, dummy, 1, None)
    assert rc != 0
    msg = L.vdt_last_error().decode()
    assert "unsupported feature-map width 130" in msg, msg
