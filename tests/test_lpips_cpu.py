"""LPIPS (VGG) without a GPU: the oracle restatement (oracle/lpips.py) against torchvision's VGG16 and a hand-computed head, the
weight files and their lookup (weights.py), and the metric's option checks (metrics.calculate_lpips)."""
import math

import pytest
import torch


def test_oracle_taps_equal_torchvision_vgg16_slices():
    import torchvision
    from oracle import lpips as ol
    from satlas_super_resolution_b200 import weights
    vgg = weights.vgg16_state(seed=4)
    net = torchvision.models.vgg16(weights=None).features.eval()
    sd = {}
    for (name, _, _), idx in zip(weights.VGG16_CONVS, weights.VGG16_TORCHVISION_INDEX):
        sd[f"{idx}.weight"], sd[f"{idx}.bias"] = vgg[f"{name}.weight"], vgg[f"{name}.bias"]
    net.load_state_dict(sd)
    x = ol.scale_input(torch.rand(2, 3, 32, 48, generator=torch.Generator().manual_seed(0)))
    with torch.no_grad():
        taps = ol.vgg16_taps(vgg, x)
        assert len(net) == 31 and isinstance(net[30], torch.nn.MaxPool2d)     # features[0:30] drops the last pool only
        for t, idx in zip(taps, ol.TAP_TORCHVISION_RELU):
            want = net[:idx + 1](x)
            assert t.shape == want.shape
            torch.testing.assert_close(t, want, rtol=1e-5, atol=1e-6)


def test_oracle_head_by_hand_and_zero_for_identical_inputs():
    from oracle import lpips as ol
    f0 = [torch.tensor([3.0, 4.0]).view(1, 2, 1, 1)]
    f1 = [torch.tensor([0.0, 2.0]).view(1, 2, 1, 1)]
    lin = {"lin0.model.1.weight": torch.tensor([0.5, 2.0]).view(1, 2, 1, 1)}
    n0, n1 = 5.0 + 1e-10, 2.0 + 1e-10
    want = 0.5 * (3 / n0 - 0 / n1) ** 2 + 2.0 * (4 / n0 - 2 / n1) ** 2
    assert math.isclose(ol.head(f0, f1, lin).item(), want, rel_tol=1e-12)
    assert ol.head(f0, f0, lin).item() == 0.0
    # the whole metric: identical images give exactly 0, and the scaling sees the bytes in the order given
    from satlas_super_resolution_b200 import weights
    vgg, lin5 = weights._lpips_seeded(1)
    img = torch.randint(0, 256, (2, 16, 16, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(2))
    assert ol.lpips(img, img, vgg, lin5) == [0.0, 0.0]
    x = ol.u8_to_input(img)
    assert torch.equal(x[:, 0], img[..., 0].float() / 255)


def test_checkpoints_in_torchvision_and_lpips_format_load(tmp_path):
    from satlas_super_resolution_b200 import weights
    raw = {}
    for (name, cin, cout), idx in zip(weights.VGG16_CONVS, weights.VGG16_TORCHVISION_INDEX):
        raw[f"features.{idx}.weight"] = torch.full((cout, cin, 3, 3), float(idx))
        raw[f"features.{idx}.bias"] = torch.full((cout,), -float(idx))
    torch.save(raw, tmp_path / "vgg16.pth")
    sd = weights.vgg16_state(pretrained_path=str(tmp_path / "vgg16.pth"))
    assert list(sd) == [f"{n}.{k}" for n, _, _ in weights.VGG16_CONVS for k in ("weight", "bias")]
    assert sd["conv3_3.weight"][0, 0, 0, 0].item() == 14.0 and sd["conv5_3.bias"][0].item() == -28.0
    assert sd["conv4_1.weight"].shape == (512, 256, 3, 3)
    lin = {f"lin{k}.model.1.weight": torch.full((1, c, 1, 1), float(k + 1)) for k, c in enumerate(weights.LPIPS_CHANNELS)}
    torch.save(lin, tmp_path / "vgg.pth")
    got = weights.lpips_lin_state(path=str(tmp_path / "vgg.pth"))
    for k, c in enumerate(weights.LPIPS_CHANNELS):
        assert got[f"lin{k}.model.1.weight"].shape == (1, c, 1, 1) and got[f"lin{k}.model.1.weight"].unique().tolist() == [k + 1.0]


def _isolate(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("TORCH_HOME", str(tmp_path / "no_hub"))
    for v in ("SSR_VGG16_PATH", "SSR_LPIPS_PATH", "SSR_LPIPS_RANDOM_SEED"):
        monkeypatch.delenv(v, raising=False)


def test_missing_lpips_weights_are_an_error_unless_random_weights_are_requested(tmp_path, monkeypatch):
    from satlas_super_resolution_b200 import weights
    _isolate(tmp_path, monkeypatch)
    with pytest.raises(FileNotFoundError) as e:
        weights.resolve_lpips_state()
    for p in weights.vgg16_search_paths() + weights.lpips_search_paths():
        assert p in str(e.value)
    with pytest.warns(RuntimeWarning):
        vgg, lin = weights.resolve_lpips_state(lpips_seed=3)
    with pytest.warns(RuntimeWarning):
        vgg2, lin2 = weights.resolve_lpips_state(lpips_seed=3)
    assert all(torch.equal(vgg[k], vgg2[k]) for k in vgg) and all(torch.equal(lin[k], lin2[k]) for k in lin)
    assert torch.equal(vgg["conv2_1.weight"], weights.vgg16_state(seed=3)["conv2_1.weight"])
    assert torch.equal(lin["lin4.model.1.weight"], weights.lpips_lin_state(seed=3)["lin4.model.1.weight"])
    w = lin["lin2.model.1.weight"]
    assert w.shape == (1, 256, 1, 1) and float(w.min()) >= 0 and float(w.max()) <= 2 / 256
    # the environment opt-in, and both files found through the environment
    monkeypatch.setenv("SSR_LPIPS_RANDOM_SEED", "3")
    assert weights.lpips_weight_source() == ("seed", 3)
    monkeypatch.delenv("SSR_LPIPS_RANDOM_SEED")
    torch.save({f"features.{i}.{k}": t for (n, _, _), i in zip(weights.VGG16_CONVS, weights.VGG16_TORCHVISION_INDEX)
                for k, t in (("weight", vgg[f"{n}.weight"]), ("bias", vgg[f"{n}.bias"]))}, tmp_path / "a.pth")
    torch.save(dict(lin), tmp_path / "b.pth")
    monkeypatch.setenv("SSR_VGG16_PATH", str(tmp_path / "a.pth"))
    with pytest.raises(FileNotFoundError):          # one of the two files alone is not enough
        weights.lpips_weight_source()
    monkeypatch.setenv("SSR_LPIPS_PATH", str(tmp_path / "b.pth"))
    assert weights.lpips_weight_source(lpips_seed=5) == ("files", str(tmp_path / "a.pth"), str(tmp_path / "b.pth"))
    vgg3, lin3 = weights.resolve_lpips_state()
    assert torch.equal(vgg3["conv5_3.weight"], vgg["conv5_3.weight"]) and torch.equal(lin3["lin0.model.1.weight"], lin["lin0.model.1.weight"])


@pytest.mark.parametrize("opt", [{}, {"lpips_model": "alexnet"}, {"lpips_model": "squeeze"}])
def test_lpips_model_other_than_vgg_is_not_implemented_before_any_lookup(tmp_path, monkeypatch, opt):
    from satlas_super_resolution_b200 import metrics as M
    from satlas_super_resolution_b200 import weights
    _isolate(tmp_path, monkeypatch)

    def no_lookup(*a, **k):
        raise AssertionError("weight lookup before the option check")
    monkeypatch.setattr(weights, "lpips_weight_source", no_lookup)
    monkeypatch.setattr(weights, "resolve_lpips_state", no_lookup)
    with pytest.raises(NotImplementedError, match="lpips_model"):
        M.calculate_lpips(None, None, **opt)
    with pytest.raises(NotImplementedError, match="lpips_model"):
        M.check_metric_opt(dict(type="calculate_lpips", **opt))
    assert "calculate_lpips" in M.METRIC_REGISTRY


def test_lpips_sizes_outside_the_built_path_raise_value_error():
    from satlas_super_resolution_b200.lpips import check_size
    check_size(128, 128)
    check_size(256, 128)
    for h, w in ((120, 120), (64, 64), (128, 120), (8, 128)):
        with pytest.raises(ValueError, match="multiples of 16"):
            check_size(h, w)
