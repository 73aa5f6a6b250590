"""Golden fixture for the data path (test infrastructure): run the UNMODIFIED reference `S2NAIPDataset`
(/root/reference/ssr/data/s2-naip_dataset.py) on the synthetic PNG tree of tests/test_data_cpu.py and record, per variant and item,
the index / chip it returned and the SHA-256 of every tensor.  `tests/test_data_cpu.py` replays the same tree and seeds through the
shard reader and compares with these digests, so the parity claim travels to machines without /root/reference.

python oracle/make_golden_data.py   # -> tests/golden/data_synthetic_tree.json
"""
import glob
import hashlib
import importlib
import json
import os
import random
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
REF = os.environ.get("SSR_REFERENCE_ROOT", "/root/reference")


def digest(sample):
    out = {"Index": sample["Index"], "Chip": sample["Chip"]}
    for k in ("lr", "hr", "old_hr"):
        if k in sample:
            t = sample[k].contiguous()
            out[k] = {"shape": list(t.shape), "sha256": hashlib.sha256(t.numpy().tobytes()).hexdigest()}
    return out


def main():
    from satlas_super_resolution_b200 import dropin
    dropin.install()                      # registry / scandir stand-ins for the absent basicsr (import-time names only)
    sys.path.insert(0, REF)
    ref_cls = importlib.import_module("ssr.data.s2-naip_dataset").S2NAIPDataset
    import test_data_cpu as t
    glob.glob = t.sorted_glob             # the test replays in name order, whatever order this file system lists
    golden = {}
    for variant in t.VARIANTS:
        root = tempfile.mkdtemp(prefix="ssr_golden_")
        t.make_tree(root, with_old=(variant == "old_hr"))
        random.seed(99)
        ds = ref_cls(t.opts(root, **t.variant_options(variant, root)))
        # the samples depend on the listing order (it fixes which random numbers each chip sees): record it
        golden[variant] = {"order": [dp[2] for dp in ds.datapoints], "items": [digest(s) for s in t.collect(ds, 1234)]}
    path = os.path.join(ROOT, "tests", "golden", "data_synthetic_tree.json")
    with open(path, "w") as fh:
        json.dump({"source": "unmodified reference S2NAIPDataset on the synthetic tree of tests/test_data_cpu.py", "variants": golden}, fh, indent=1)
    print("wrote", path, {k: len(v['items']) for k, v in golden.items()})


if __name__ == "__main__":
    main()
