"""Golden values for the checks against the reference's own code (test infrastructure), so the tests need no reference checkout:

    tests/golden/ref_modules.pt             SSR_RRDBNet / SSR_UNetDiscriminatorSN (through oracle/ref_shim.py): one generator output,
                                            the key schema and the default-init spread
    tests/golden/format_s2naip_data.pt      ssr/utils/infer_utils.py format_s2naip_data on the seeded input of tests/test_host_cpu.py
    tests/golden/dropin_infer_example.json  the arch modules ssr/archs/__init__.py scans, the options of ssr/options/infer_example.yml
                                            that ssr/utils/model_utils.build_network reads, and the reference generator's state_dict keys

Run from the repo root with the reference checkout at $SSR_REFERENCE_ROOT:  python -m oracle.make_golden_ref
"""
import importlib.util
import json
import os
import random
import subprocess
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import nets, ref_shim  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

# the reference's scanner and option loader need the drop-in stand-ins for basicsr, which change sys.modules: own interpreter
SCANNER = r'''
import json, os, sys
sys.path.insert(0, %r)
from satlas_super_resolution_b200 import dropin
dropin.install(reference_root=%r)
import ssr.archs
from ssr.utils.options import yaml_load
opt = yaml_load(%r)
print(json.dumps({"arch_modules": ssr.archs.arch_filenames,
                  "opt": {"scale": opt["scale"], "n_lr_images": opt["n_lr_images"], "network_g": opt["network_g"]}}))
'''


def modules():
    RRDB, UNetD = ref_shim.reference_archs()
    sd = nets.rrdbnet_init(24, 3, num_block=1, seed=5)
    m = RRDB(num_in_ch=24, num_out_ch=3, num_block=1)
    m.load_state_dict(sd, strict=True)
    x = torch.rand(1, 24, 32, 32, generator=torch.Generator().manual_seed(6))
    with torch.no_grad():
        y = m.eval()(x)
    torch.manual_seed(0)
    g2 = RRDB(num_in_ch=24, num_out_ch=3, num_block=2).state_dict()
    d = UNetD(num_in_ch=27).state_dict()
    std_keys = ("body.0.rdb1.conv1.weight", "conv_first.weight", "body.1.rdb3.conv5.weight")
    torch.save({"sd_seed": 5, "x_seed": 6, "y": y.clone(),
                "g1_shapes": [(k, list(v.shape)) for k, v in m.state_dict().items()],
                "g2_shapes": [(k, list(v.shape)) for k, v in g2.items()], "g2_std": {k: g2[k].std().item() for k in std_keys},
                "g2_bias_abs_max": g2["body.0.rdb2.conv3.bias"].abs().max().item(),
                "d_shapes": [(k, list(v.shape)) for k, v in d.items()]}, os.path.join(OUT, "ref_modules.pt"))
    return RRDB


def format_s2naip():
    sys.modules.setdefault("skimage", types.ModuleType("skimage"))         # imported by infer_utils, not used by this function
    sys.modules.setdefault("skimage.io", types.ModuleType("skimage.io"))
    spec = importlib.util.spec_from_file_location("_ref_infer_utils", os.path.join(ref_shim.REFERENCE_ROOT, "ssr", "utils", "infer_utils.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_host_cpu import format_s2naip_input
    random.seed(5)
    want, first = mod.format_s2naip_data(format_s2naip_input(), 8, "cpu")
    u8 = (want * 255).round().to(torch.uint8)              # the frames are bytes / 255: stored as the bytes, a quarter of the size
    assert torch.equal(u8.float() / 255, want)
    torch.save({"random_seed": 5, "n_s2_images": 8, "s2_tensor_u8": u8, "s2_image": torch.from_numpy(np.ascontiguousarray(first))},
               os.path.join(OUT, "format_s2naip_data.pt"))


def dropin_options(RRDB):
    ref = ref_shim.REFERENCE_ROOT
    code = SCANNER % (ROOT, ref, os.path.join(ref, "ssr", "options", "infer_example.yml"))
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True)
    gold = json.loads(res.stdout.strip().splitlines()[-1])
    opt, net = gold["opt"], gold["opt"]["network_g"]
    # ssr/utils/model_utils.py build_network, with the reference's own class
    m = RRDB(num_in_ch=int(opt["n_lr_images"]) * 3, num_out_ch=3, num_feat=int(net["num_feat"]), num_block=int(net["num_block"]),
             num_grow_ch=int(net["num_grow_ch"]), scale=int(opt["scale"]))
    gold["state_dict_keys"] = list(m.state_dict().keys())
    with open(os.path.join(OUT, "dropin_infer_example.json"), "w") as fh:
        json.dump(gold, fh, indent=1)


def main():
    RRDB = modules()
    format_s2naip()
    dropin_options(RRDB)
    print("golden fixtures written to", OUT)


if __name__ == "__main__":
    main()
