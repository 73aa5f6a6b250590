"""CPU tests of the packed-shard data path (satlas_super_resolution_b200/data.py, SURVEY.md 8f row 2).

A small synthetic S2-NAIP tree (PNG files, written with cv2) exercises every branch of the sample assembly: a NAIP chip with a
black pixel (rejected), Sentinel-2 frames with black pixels (used only to fill up), a chip with too few frames, a missing band
file, the random-crop augmentation, `train_samples` sub-sampling and `old_naip_path`.  With the same `random` seed
  * the shard reader returns the same tensors as the PNG reader of the same class, and
  * both return what the UNMODIFIED reference `S2NAIPDataset` returned (tests/golden/data_synthetic_tree.json), item by item,
    including the indices it skips to.
"""
import glob
import os
import random

import numpy as np
import pytest
import torch

cv2 = pytest.importorskip("cv2")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_S2 = 4
_glob = glob.glob


def sorted_glob(*args, **kwargs):
    """glob.glob in name order.  The datasets list chips in glob order, and the order fixes which random numbers each chip
    draws; directory order differs between file systems, so the fixture is recorded and replayed in name order."""
    return sorted(_glob(*args, **kwargs))


def _write_png(path, chw):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    a = np.ascontiguousarray(np.transpose(chw, (1, 2, 0)))
    assert cv2.imwrite(path, a[..., ::-1] if a.shape[2] == 3 else a[..., 0])


def make_tree(root, with_old=False):
    rng = np.random.default_rng(5)
    chips = [f"{10 + i}_{20 + i}" for i in range(7)]
    for i, chip in enumerate(chips):
        hr = rng.integers(1, 256, (3, 128, 128), dtype=np.uint8)
        if i == 2:
            hr[:, 5, 7] = 0                                   # a black pixel: the reference skips this datapoint
        _write_png(os.path.join(root, "naip", "2020", chip, f"{chip}.png"), hr)
        if with_old:
            _write_png(os.path.join(root, "old_naip", "2017", f"{chip}.png"), rng.integers(1, 256, (3, 128, 128), dtype=np.uint8))
        # chip 4 has fewer frames than requested; chip 3 (no b08.png) has exactly n_s2_images frames -- the reference's zero
        # stand-in for a missing band has n_s2_images frames, so it only concatenates with a series of that length
        T = 3 if i == 4 else (N_S2 if i == 3 else 7)
        tci = rng.integers(1, 256, (3, T * 32, 32), dtype=np.uint8)
        if i in (1, 5):
            for t in ((0, 2, 3, 6) if i == 1 else (1,)):      # chip 1: only 3 clean frames left -> bad ones fill up
                tci[:, t * 32 + 3, 4] = 0
        _write_png(os.path.join(root, "s2", chip, "tci.png"), tci)
        if i != 3:                                            # chip 3 lacks the extra band: zeros of n_s2_images frames
            _write_png(os.path.join(root, "s2", chip, "b08.png"), rng.integers(1, 256, (1, T * 32, 32), dtype=np.uint8))
    return chips


def opts(root, **kw):
    o = dict(phase="train", n_s2_images=N_S2, scale=4, sentinel2_path=os.path.join(root, "s2"), naip_path=os.path.join(root, "naip"),
             s2_bands=["b08", "tci"])
    o.update(kw)
    return o


def collect(ds, seed):
    random.seed(seed)
    out = []
    for i in range(len(ds)):
        s = ds[i]
        out.append({k: (v.clone() if torch.is_tensor(v) else v) for k, v in s.items()})
    return out


def assert_same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x["Index"] == y["Index"] and x["Chip"] == y["Chip"] and x["Phase"] == y["Phase"]
        for k in ("lr", "hr", "old_hr"):
            assert (k in x) == (k in y)
            if k in x:
                assert x[k].dtype == torch.uint8 and x[k].shape == y[k].shape and torch.equal(x[k], y[k]), k


VARIANTS = ["plain", "rand_crop", "subset", "old_hr"]


def variant_options(variant, root):
    return {"plain": {}, "rand_crop": {"rand_crop": True}, "subset": {"train_samples": 5},
            "old_hr": {"old_naip_path": os.path.join(root, "old_naip")}}[variant]


def check_against_golden(variant, samples, order):
    """digests recorded from the unmodified reference dataset by oracle/make_golden_data.py, chips listed in name order"""
    import hashlib
    import json
    with open(os.path.join(ROOT, "tests", "golden", "data_synthetic_tree.json")) as fh:
        gold = json.load(fh)["variants"][variant]
    assert gold["order"] == order
    want = gold["items"]
    assert len(want) == len(samples)
    for w, s in zip(want, samples):
        assert w["Index"] == s["Index"] and w["Chip"] == s["Chip"]
        for k in ("lr", "hr", "old_hr"):
            assert (k in w) == (k in s)
            if k in w:
                assert w[k]["shape"] == list(s[k].shape)
                assert w[k]["sha256"] == hashlib.sha256(s[k].contiguous().numpy().tobytes()).hexdigest(), (variant, s["Chip"], k)


@pytest.mark.parametrize("variant", VARIANTS)
def test_shard_reader_matches_png_reader_and_reference(tmp_path, monkeypatch, variant):
    from satlas_super_resolution_b200.data import S2NAIPShardDataset, pack_s2naip
    monkeypatch.setattr(glob, "glob", sorted_glob)
    root = str(tmp_path)
    make_tree(root, with_old=(variant == "old_hr"))
    extra = variant_options(variant, root)
    prefix = os.path.join(root, "shard0")
    assert pack_s2naip(opts(root, **extra), prefix) == 7

    def build(cls, **kw):
        random.seed(99)                                       # `train_samples` draws from the global state at construction
        return cls(opts(root, **extra, **kw))

    png = collect(build(S2NAIPShardDataset), 1234)
    shard_ds = build(S2NAIPShardDataset, shard_path=prefix)
    shard = collect(shard_ds, 1234)
    assert_same(png, shard)
    s0 = shard[0]
    assert s0["lr"].shape == (N_S2 * 4, 32, 32) and s0["hr"].shape == (3, 128, 128)
    # the datapoint with the black NAIP pixel is never returned; the one with too few frames neither
    assert all(s["Chip"] not in ("12_22", "14_24") for s in shard)
    check_against_golden(variant, shard, [rec["chip"] for rec in shard_ds.datapoints])


def test_frame_choice_prefers_clean_frames(tmp_path):
    from satlas_super_resolution_b200.data import S2NAIPShardDataset, has_black_pixels, pack_s2naip
    root = str(tmp_path)
    make_tree(root)
    prefix = os.path.join(root, "s")
    pack_s2naip(opts(root), prefix)
    ds = S2NAIPShardDataset(opts(root, shard_path=prefix))
    random.seed(3)
    by_chip = {}
    for i in range(len(ds)):
        s = ds[i]
        by_chip.setdefault(s["Chip"], s)
    # chip 15_25 has one bad frame out of 7: the 4 chosen frames are all clean (channels: t * 4 + c, TCI first)
    lr = by_chip["15_25"]["lr"].view(N_S2, 4, 32, 32)
    assert not any(has_black_pixels(f[:3]) for f in lr)
    # chip 11_21 has only 3 clean frames: exactly one chosen frame carries a black pixel
    lr = by_chip["11_21"]["lr"].view(N_S2, 4, 32, 32)
    assert sum(bool(has_black_pixels(f[:3])) for f in lr) == 1
    # chip 13_23 lacks b08.png: that channel is all zeros, TCI is not
    lr = by_chip["13_23"]["lr"].view(N_S2, 4, 32, 32)
    assert lr[:, 3].abs().max() == 0 and lr[:, :3].max() > 0


def test_shard_guards_and_batcher(tmp_path):
    from satlas_super_resolution_b200.data import PinnedBatcher, S2NAIPShardDataset, pack_s2naip
    from satlas_super_resolution_b200.registry import DATASET_REGISTRY
    assert DATASET_REGISTRY.get("S2NAIPShardDataset") is S2NAIPShardDataset
    root = str(tmp_path)
    make_tree(root)
    prefix = os.path.join(root, "s")
    pack_s2naip(opts(root), prefix)
    with pytest.raises(ValueError, match="bands"):
        S2NAIPShardDataset(opts(root, shard_path=prefix, s2_bands=["tci"]))
    with pytest.raises(ValueError, match="old_naip_path"):
        S2NAIPShardDataset(opts(root, shard_path=prefix, old_naip_path=os.path.join(root, "nowhere")))
    with pytest.raises(NotImplementedError):
        S2NAIPShardDataset(opts(root, shard_path=prefix, osm_objs_path="x.json"))
    ds = S2NAIPShardDataset(opts(root, shard_path=prefix))
    random.seed(0)
    pb = PinnedBatcher(ds, 3, pin=False)
    random.seed(7)
    b = pb.batch([0, 1, 5])
    random.seed(7)
    want = [ds[i] for i in (0, 1, 5)]
    assert b["lr"].shape == (3, N_S2 * 4, 32, 32) and b["hr"].shape == (3, 3, 128, 128)
    for i, s in enumerate(want):
        assert torch.equal(b["lr"][i], s["lr"]) and torch.equal(b["hr"][i], s["hr"])
    w = ds.get_tile_weight_sampler({"10_20": 5.0})
    assert len(list(iter(w))) == len(ds)
    # the `tile_weights` option (a JSON of {chip: weight}; read by nothing in the reference) wired to the sampler, and the sampler to the batcher
    import json
    from satlas_super_resolution_b200.data import build_train_sampler
    assert build_train_sampler(ds, {"use_shuffle": True}) is None
    chips = [rec["naip"].split("/")[-1][:-4] for rec in ds.datapoints]
    wpath = os.path.join(root, "weights.json")
    json.dump({chips[0]: 1e9}, open(wpath, "w"))
    with pytest.raises(ValueError, match="use_shuffle"):
        build_train_sampler(ds, {"tile_weights": wpath, "use_shuffle": True})
    sampler = build_train_sampler(ds, {"tile_weights": wpath, "use_shuffle": False})
    np.random.seed(0)
    drawn = list(iter(sampler))
    assert len(drawn) == len(ds) and drawn.count(0) >= len(ds) - 1          # weight 1e9 against 1: (almost) always datapoint 0
    assert [float(x) for x in sampler.weights] == [1e9] + [1.0] * (len(ds) - 1)
    np.random.seed(0)
    random.seed(11)
    got = list(pb.batches(sampler))
    assert len(got) == len(ds) // 3 and all(b["lr"].shape[0] == 3 for b in got)
