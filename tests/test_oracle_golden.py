"""CPU tests: the oracle (oracle/*.py) reproduces the golden vectors that tests/golden/make_golden.py produced by
running the reference's own classes on the same name-seeded weights and inputs.  Both sides run in float64 and are
compared at rtol 1e-9 / atol 1e-10 (reference_golden_f64.npz): the CPU's vector width and thread count change the
summation order and move results by about 1e-14, while in fp32 they move them by about 1e-6, so an fp32 comparison
would fail on other machines.  reference_golden.json holds the shapes and counts and the reference's fp32 outputs, which
must agree with the float64 run to fp32 accuracy."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import cases
from oracle.adapter import ControlNetAdapter, ControlNetRouter
from oracle.blocks import ResnetBlock2D
from oracle.controlnet import ControlNetModel, MultiControlNetModel
from oracle.weights import fingerprint, seeded_init_, seeded_tensor

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
GOLD = json.load(open(os.path.join(GOLDEN, "reference_golden.json")))
GOLD64 = dict(np.load(os.path.join(GOLDEN, "reference_golden_f64.npz")))  # key -> [mean, std, absmax, samples...]
torch.set_grad_enabled(False)


def assert_fp(t, key, rtol=1e-9, atol=1e-10):
    """`key` is the fingerprint's path in the golden data, e.g. "adapter_sdxl.down.3"."""
    gold = GOLD
    for k in key.split("."):
        gold = gold[int(k)] if isinstance(gold, list) else gold[k]
    got = fingerprint(t, len(gold["samples"]))
    assert got["shape"] == gold["shape"]
    samples = torch.tensor(got["samples"], dtype=torch.float64)
    mean, _, absmax = (float(v) for v in GOLD64[key][:3])
    torch.testing.assert_close(samples, torch.from_numpy(GOLD64[key][3:]), rtol=rtol, atol=atol)
    assert abs(got["mean"] - mean) <= atol + rtol * abs(mean) + rtol * absmax
    assert abs(got["absmax"] - absmax) <= atol + rtol * absmax
    torch.testing.assert_close(samples, torch.tensor(gold["samples"], dtype=torch.float64), rtol=0,
                               atol=1e-4 * gold["absmax"])


def test_adapter_sdxl_matches_reference():
    m = seeded_init_(ControlNetAdapter(**cases.ADAPTER_SDXL_KW), seed=1).double().eval()
    down, mid = m(**cases.to_double(cases.adapter_sdxl_inputs()))
    assert mid is None and GOLD["adapter_sdxl"]["mid"] is None
    assert len(down) == 12
    for i, t in enumerate(down):
        assert_fp(t, f"adapter_sdxl.down.{i}")
    # blocks 9..11 are not selected for SDXL: new zero tensors of the input shape (ctrl_adapter.py:193)
    assert all(float(t.abs().max()) == 0.0 for t in down[9:])


def test_adapter_video_matches_reference():
    m = seeded_init_(ControlNetAdapter(**cases.ADAPTER_VIDEO_KW), seed=2).double().eval()
    down, mid = m(**cases.to_double(cases.adapter_video_inputs()))
    for i, t in enumerate(down):
        assert_fp(t, f"adapter_video.down.{i}")
    assert_fp(mid, "adapter_video.mid")


def test_router_matches_reference():
    r = seeded_init_(ControlNetRouter(**cases.ROUTER_KW), seed=3).double().eval()
    dw, mw = r(sparse_mask=cases.ROUTER_MASK)
    assert_fp(dw, "router.down")
    assert_fp(mw, "router.mid")
    assert dw.shape == (12, 7) and mw.shape == (7,)
    # masked experts get (numerically) zero weight
    assert float(dw[:, [2, 4, 5, 6]].max()) == 0.0
    dw, mw = r(sparse_mask=None)
    assert_fp(dw, "router_nomask.down")
    assert_fp(mw, "router_nomask.mid")


def test_controlnet_matches_reference():
    cn = seeded_init_(ControlNetModel(**cases.CONTROLNET_KW), seed=4).double().eval()
    inp = cases.to_double(cases.controlnet_inputs())
    down, mid = cn(**inp)
    assert len(down) == 12
    for i, t in enumerate(down):
        assert_fp(t, f"controlnet.down.{i}")
    assert_fp(mid, "controlnet.mid")
    down, mid = cn(**{**inp, "skip_conv_in": True, "conditioning_scale": 0.75})
    for i, t in enumerate(down):
        assert_fp(t, f"controlnet_skip_conv_in.down.{i}")
    # MultiControlNet: zip() truncation to the number of provided images, list outputs (multicontrolnet.py:66-99)
    multi = MultiControlNetModel([cn, cn, cn])
    conds = [inp["controlnet_cond"], torch.flip(inp["controlnet_cond"], dims=[3])]
    dl, ml = multi(inp["sample"], inp["timestep"], inp["encoder_hidden_states"], conds, [1.0, 0.5, 0.25], return_dict=False)
    assert len(dl) == GOLD["multicontrolnet"]["n_nets_run"] == 2
    for i, t in enumerate(dl[1]):
        assert_fp(t, f"multicontrolnet.down1.{i}")
    assert_fp(ml[1], "multicontrolnet.mid1")


def test_resnet_upsample_output_size_matches_reference():
    rb = seeded_init_(ResnetBlock2D(in_channels=320, out_channels=320, temb_channels=320, eps=1e-6,
                                    use_in_shortcut=True, up=True), seed=5).double().eval()
    x = seeded_tensor("rb_x", (2, 320, 6, 5), 5, dtype=torch.float64)
    temb = seeded_tensor("rb_temb", (2, 320), 5, dtype=torch.float64)
    assert_fp(rb(x, temb, output_size=(12, 10)), "resnet_up")
    assert_fp(rb(x, temb, output_size=(9, 8)), "resnet_up_odd")


# ---- self-consistency checks that stand in for the missing upstream KATs (SURVEY.md section 8c) ----
def test_timesteps_closed_form():
    from oracle.blocks import Timesteps
    import math
    t = torch.tensor([0.0, 1.0, 500.0, 999.0])
    emb = Timesteps(320, True, 0)(t)
    k = torch.arange(160, dtype=torch.float64)
    freq = torch.exp(-math.log(10000.0) * k / 160)
    arg = t.double()[:, None] * freq[None]
    ref = torch.cat([torch.cos(arg), torch.sin(arg)], -1)
    torch.testing.assert_close(emb.double(), ref, rtol=0, atol=2e-4)


def test_attention_matches_explicit_softmax_fp64():
    from oracle.blocks import Attention
    a = seeded_init_(Attention(query_dim=64, heads=2, dim_head=32), 9).double()
    x = seeded_tensor("att_x", (2, 10, 64), 9).double()
    q, k, v = a.to_q(x), a.to_k(x), a.to_v(x)
    q, k, v = (t.view(2, 10, 2, 32).transpose(1, 2) for t in (q, k, v))
    p = torch.softmax(q @ k.transpose(-1, -2) / 32 ** 0.5, -1)
    ref = a.to_out[0]((p @ v).transpose(1, 2).reshape(2, 10, 64))
    torch.testing.assert_close(a(x), ref, rtol=1e-10, atol=1e-12)


def test_sdxl_unet_param_count_and_adapter_wiring():
    """2 567 463 684 parameters = the published SDXL-base UNet size; 361 279 120 = SD1.5 ControlNet."""
    from oracle.unet_sdxl import UNet2DConditionModel
    with torch.device("meta"):
        u = UNet2DConditionModel()
        c = ControlNetModel(**cases.CONTROLNET_KW)
    assert sum(p.numel() for p in u.parameters()) == 2567463684
    assert sum(p.numel() for p in c.parameters()) == 361279120


def test_unet_svd_matches_reference():
    """Reduced-width SVD UNet (same block types / depths as the released model) incl. the reference's 5-D residual
    injection with zip truncation and the mid residual (svd/.../unet_spatio_temporal_condition.py:457-471, 485-490)."""
    from oracle.unet_svd import UNetSpatioTemporalConditionModel
    u = seeded_init_(UNetSpatioTemporalConditionModel(**cases.UNET_SVD_SMALL_KW), seed=11).double().eval()
    assert sum(p.numel() for p in u.parameters()) == GOLD["unet_svd_small"]["n_params"]
    assert_fp(u(**cases.to_double(cases.unet_svd_inputs(with_residuals=True)))[0], "unet_svd_small.with_residuals")
    assert_fp(u(**cases.to_double(cases.unet_svd_inputs(with_residuals=False)))[0], "unet_svd_small.plain")


def test_unet_i2vgen_matches_reference():
    """Reduced-width I2VGen-XL UNet incl. the residual injection (i2vgen_xl/.../unet_i2vgen_xl.py:681-695, 709-714)."""
    from oracle.unet_i2vgen import I2VGenXLUNet
    u = seeded_init_(I2VGenXLUNet(**cases.UNET_I2VGEN_SMALL_KW), seed=12).double().eval()
    assert sum(p.numel() for p in u.parameters()) == GOLD["unet_i2vgen_small"]["n_params"]
    assert_fp(u(**cases.to_double(cases.unet_i2vgen_small_inputs(with_residuals=True)))[0],
              "unet_i2vgen_small.with_residuals")
    assert_fp(u(**cases.to_double(cases.unet_i2vgen_small_inputs(with_residuals=False)))[0], "unet_i2vgen_small.plain")
