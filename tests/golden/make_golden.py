"""Generates tests/golden/reference_golden.json by running the REAL reference classes from /root/reference
(model/ctrl_adapter.py, model/adapter_spatial_temporal.py, model/resnet_block_2d.py, model/ctrl_router.py,
controlnet/controlnet.py, controlnet/multicontrolnet.py, i2vgen_xl/models/unets/unet_i2vgen_xl.py,
svd/models/unets/unet_spatio_temporal_condition.py) on CPU, in fp32 (reference_golden.json: shapes, counts and
fingerprints) and in float64 (reference_golden_f64.npz: the fingerprints that the oracle is held to, since in float64
they do not depend on the summation order of the CPU that computes them).

The reference imports `diffusers`, which is not installed here; oracle/diffusers_shim provides the needed module
paths backed by the restated blocks of oracle/blocks.py.  So these vectors pin the reference's own (in-repo) layer of
the hot path; the third-party diffusers layer underneath is restated, not pinned (see oracle/blocks.py header).

Run in the build container only (needs /root/reference):   python tests/golden/make_golden.py
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "diffusers_shim"))

from oracle import cases  # noqa: E402
from oracle.weights import fingerprint, seeded_init_, seeded_tensor  # noqa: E402
import oracle.blocks  # noqa: E402,F401  (everything the shim needs from this repo is imported before ROOT leaves sys.path)

# The repo root also holds drop-in packages named like the reference's (model/, controlnet/, i2vgen_xl/, sdxl/, svd/);
# they are regular packages and would shadow the reference's namespace packages whatever the path order.  From here on
# only /root/reference (and the diffusers shim) may resolve those names.
sys.path[:] = [p for p in sys.path if os.path.abspath(p or os.getcwd()) != ROOT]
for _name in [m for m in sys.modules if m.split(".")[0] in ("model", "controlnet", "i2vgen_xl", "sdxl", "svd", "utils")]:
    del sys.modules[_name]
sys.path.insert(0, "/root/reference")

torch.set_grad_enabled(False)
torch.manual_seed(0)

from controlnet.controlnet import ControlNetModel  # noqa: E402  (reference)
from controlnet.multicontrolnet import MultiControlNetModel  # noqa: E402
from model.ctrl_adapter import ControlNetAdapter  # noqa: E402
from model.ctrl_router import ControlNetRouter  # noqa: E402
from model.resnet_block_2d import ResnetBlock2D  # noqa: E402
assert ControlNetAdapter.__module__ == "model.ctrl_adapter" and "/root/reference/" in sys.modules[ControlNetAdapter.__module__].__file__

out = {"_meta": {"reference": "HL-hanlin/Ctrl-Adapter @ /root/reference", "torch": torch.__version__,
                 "note": "fp32 CPU outputs of the reference's own classes over oracle/diffusers_shim"}}


def fp_list(ts):
    return [fingerprint(t) for t in ts]


def generate(dtype):
    """Fingerprints of every case with the modules and inputs in `dtype`."""
    cast = cases.to_double if dtype == torch.float64 else (lambda x: x)
    out = {}
    # --- G1: ControlNetAdapter, SDXL configuration ------------------------------------------------------
    m = seeded_init_(ControlNetAdapter(**cases.ADAPTER_SDXL_KW), seed=1).to(dtype).eval()
    down, mid = m(**cast(cases.adapter_sdxl_inputs()))
    out["adapter_sdxl"] = {"down": fp_list(down), "mid": None if mid is None else fingerprint(mid)}
    print("adapter_sdxl done", [tuple(d.shape) for d in down][:4])
    del m

    # --- G2: ControlNetAdapter, video configuration (spatial+temporal resnet & transformer, A-D + M) -----
    m = seeded_init_(ControlNetAdapter(**cases.ADAPTER_VIDEO_KW), seed=2).to(dtype).eval()
    down, mid = m(**cast(cases.adapter_video_inputs()))
    out["adapter_video"] = {"down": fp_list(down), "mid": fingerprint(mid)}
    print("adapter_video done")
    del m

    # --- G3: router (the reference calls .cuda() unconditionally, ctrl_router.py:21,38 -> neutralised on CPU) -----
    torch.Tensor.cuda = lambda self, *a, **k: self
    r = seeded_init_(ControlNetRouter(**cases.ROUTER_KW), seed=3).to(dtype).eval()
    dw, mw = r(sparse_mask=cases.ROUTER_MASK)
    out["router"] = {"down": fingerprint(dw, 1024), "mid": fingerprint(mw, 1024)}
    dw2, mw2 = r(sparse_mask=None)
    out["router_nomask"] = {"down": fingerprint(dw2, 1024), "mid": fingerprint(mw2, 1024)}
    print("router done", dw.shape, mw.shape)

    # --- G4: ControlNetModel (+ skip_conv_in variant) and MultiControlNetModel list semantics -------------------
    cn = seeded_init_(ControlNetModel(**cases.CONTROLNET_KW), seed=4).to(dtype).eval()
    inp = cast(cases.controlnet_inputs())
    down, mid = cn(**inp)
    out["controlnet"] = {"down": fp_list(down), "mid": fingerprint(mid)}
    down, mid = cn(**{**inp, "skip_conv_in": True, "conditioning_scale": 0.75})
    out["controlnet_skip_conv_in"] = {"down": fp_list(down), "mid": fingerprint(mid)}
    multi = MultiControlNetModel([cn, cn, cn])
    conds = [inp["controlnet_cond"], torch.flip(inp["controlnet_cond"], dims=[3])]
    dl, ml = multi(inp["sample"], inp["timestep"], inp["encoder_hidden_states"], conds, [1.0, 0.5, 0.25],
                   return_dict=False)
    out["multicontrolnet"] = {"n_nets_run": len(dl), "down1": fp_list(dl[1]), "mid1": fingerprint(ml[1])}
    print("controlnet done")
    del cn, multi

    # --- G5: the reference's ResnetBlock2D copy with up-sampling to an explicit output_size --------------------
    rb = seeded_init_(ResnetBlock2D(in_channels=320, out_channels=320, temb_channels=320, eps=1e-6,
                                    use_in_shortcut=True, up=True), seed=5).to(dtype).eval()
    x = seeded_tensor("rb_x", (2, 320, 6, 5), 5, dtype=dtype)
    temb = seeded_tensor("rb_temb", (2, 320), 5, dtype=dtype)
    out["resnet_up"] = fingerprint(rb(x, temb, output_size=(12, 10)))
    out["resnet_up_odd"] = fingerprint(rb(x, temb, output_size=(9, 8)))
    print("resnet done")

    # --- G6: the two video UNets with the reference's residual-injection additions (reduced width, real block types) --
    from i2vgen_xl.models.unets.unet_i2vgen_xl import I2VGenXLUNet  # (reference)
    from svd.models.unets.unet_spatio_temporal_condition import UNetSpatioTemporalConditionModel  # (reference)

    u = seeded_init_(UNetSpatioTemporalConditionModel(**cases.UNET_SVD_SMALL_KW), seed=11).to(dtype).eval()
    out["unet_svd_small"] = {
        "with_residuals": fingerprint(u(**cast(cases.unet_svd_inputs(with_residuals=True)), return_dict=False)[0]),
        "plain": fingerprint(u(**cast(cases.unet_svd_inputs(with_residuals=False)), return_dict=False)[0]),
        "n_params": sum(p.numel() for p in u.parameters())}
    print("unet_svd_small done")
    del u
    u = seeded_init_(I2VGenXLUNet(**cases.UNET_I2VGEN_SMALL_KW), seed=12).to(dtype).eval()
    out["unet_i2vgen_small"] = {
        "with_residuals": fingerprint(u(**cast(cases.unet_i2vgen_small_inputs(with_residuals=True)),
                                        return_dict=False)[0]),
        "plain": fingerprint(u(**cast(cases.unet_i2vgen_small_inputs(with_residuals=False)), return_dict=False)[0]),
        "n_params": sum(p.numel() for p in u.parameters())}
    print("unet_i2vgen_small done")
    del u
    return out


def flatten(x, key, flat):
    """{"adapter_sdxl.down.3": [mean, std, absmax, samples...], ...} of a generate() result."""
    if isinstance(x, dict) and "samples" in x:
        flat[key] = np.array([x["mean"], x["std"], x["absmax"]] + x["samples"], dtype=np.float64)
    elif isinstance(x, dict):
        for k, v in x.items():
            flatten(v, f"{key}.{k}" if key else k, flat)
    elif isinstance(x, list):
        for i, v in enumerate(x):
            flatten(v, f"{key}.{i}", flat)
    return flat


HERE = os.path.dirname(os.path.abspath(__file__))
out.update(generate(torch.float32))
path = os.path.join(HERE, "reference_golden.json")
with open(path, "w") as f:
    json.dump(out, f)
print("wrote", path, os.path.getsize(path), "bytes")
path = os.path.join(HERE, "reference_golden_f64.npz")
np.savez_compressed(path, **flatten(generate(torch.float64), "", {}))
print("wrote", path, os.path.getsize(path), "bytes")
