"""CPU tests of the drop-in boundary: registry surface, constructor signatures, state_dict key schema, and that the
reference's package scanners and builders return OUR classes."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_registry_surface_and_schema():
    from oracle import nets
    from satlas_super_resolution_b200 import archs, losses, models, registry  # noqa: F401
    assert registry.ARCH_REGISTRY.get("SSR_RRDBNet") is archs.SSR_RRDBNet
    assert registry.ARCH_REGISTRY.get("SSR_UNetDiscriminatorSN") is archs.SSR_UNetDiscriminatorSN
    assert registry.MODEL_REGISTRY.get("SSRESRGANModel") is models.SSRESRGANModel
    for n in ("L1Loss", "GANLoss", "PerceptualLoss"):
        assert n in registry.LOSS_REGISTRY
    g = registry.build_network(dict(type="SSR_RRDBNet", num_in_ch=24, num_out_ch=3, num_feat=64, num_block=2, num_grow_ch=32))
    ref_sd = nets.rrdbnet_init(24, 3, num_block=2)
    assert list(g.state_dict().keys()) == list(ref_sd.keys())
    assert all(g.state_dict()[k].shape == v.shape for k, v in ref_sd.items())
    g.load_state_dict(ref_sd, strict=True)
    d = registry.build_network(dict(type="SSR_UNetDiscriminatorSN", num_in_ch=27, num_feat=64, skip_connection=True))
    dref = nets.unet_disc_init(27)
    assert list(d.state_dict().keys()) == list(dref.keys())
    d.load_state_dict(dref, strict=True)
    assert sum(p.numel() for p in registry.build_network(dict(type="SSR_RRDBNet", num_in_ch=24, num_out_ch=3)).parameters()) == 16_710_083
    assert sum(p.numel() for p in d.parameters()) == 4_390_721
    # the init distributions follow the reference: RDB convs ~ N(0, (0.1*sqrt(2/fan_in))^2), zero bias
    w = g.state_dict()["body.0.rdb1.conv1.weight"]
    assert abs(w.std().item() / (0.1 * (2.0 / (64 * 9)) ** 0.5) - 1) < 0.05
    assert g.state_dict()["body.1.rdb2.conv4.bias"].abs().max() == 0


def test_no_cpu_fallback():
    from satlas_super_resolution_b200 import archs
    g = archs.SSR_RRDBNet(3, 3, num_block=1)
    with pytest.raises(RuntimeError, match="no CPU path"):
        g(torch.rand(1, 3, 32, 32))
    d = archs.SSR_UNetDiscriminatorSN(3)
    with pytest.raises(RuntimeError, match="no CPU path"):
        d(torch.rand(1, 3, 64, 64))


def test_unsupported_options_fail_loudly():
    from satlas_super_resolution_b200 import losses
    with pytest.raises(NotImplementedError):
        losses.GANLoss("hinge")
    with pytest.raises(NotImplementedError):
        losses.PerceptualLoss({"conv5_4": 1.0}, style_weight=1.0)


def test_reference_scanners_pick_up_our_classes():
    """run in a subprocess: dropin.install(), then what the reference's arch scanner (ssr/archs/__init__.py) and
    ssr/utils/model_utils.build_network do with ssr/options/infer_example.yml.  The scanned module names, the options and the
    reference generator's state_dict keys were recorded from the reference (oracle/make_golden_ref.py)."""
    code = r'''
import importlib, json, sys
sys.path.insert(0, %r)
import satlas_super_resolution_b200.dropin as dropin
dropin.install()
from basicsr.utils.registry import ARCH_REGISTRY
from satlas_super_resolution_b200 import archs
with open(%r) as fh:
    gold = json.load(fh)
assert {"rrdbnet_arch", "discriminator_arch"} <= set(gold["arch_modules"])
mods = {n: importlib.import_module(f"ssr.archs.{n}") for n in ("rrdbnet_arch", "discriminator_arch")}   # as the scanner imports them
assert mods["rrdbnet_arch"].SSR_RRDBNet is archs.SSR_RRDBNet, "the scanner does not import the engine module"
assert mods["discriminator_arch"].SSR_UNetDiscriminatorSN is archs.SSR_UNetDiscriminatorSN
assert ARCH_REGISTRY.get("SSR_RRDBNet") is archs.SSR_RRDBNet, "registry does not hold the engine class"
assert ARCH_REGISTRY.get("SSR_UNetDiscriminatorSN") is archs.SSR_UNetDiscriminatorSN
opt, net = gold["opt"], gold["opt"]["network_g"]
m = mods["rrdbnet_arch"].SSR_RRDBNet(num_in_ch=int(opt["n_lr_images"]) * 3, num_out_ch=3, num_feat=int(net["num_feat"]),
                                     num_block=int(net["num_block"]), num_grow_ch=int(net["num_grow_ch"]), scale=int(opt["scale"]))
assert type(m) is archs.SSR_RRDBNet and m.num_in_ch == int(opt["n_lr_images"]) * 3
assert list(m.state_dict().keys()) == gold["state_dict_keys"], "checkpoints of the reference generator would not load"
print("OK", len(m.state_dict()))
''' % (ROOT, os.path.join(ROOT, "tests", "golden", "dropin_infer_example.json"))
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "OK 702" in res.stdout
