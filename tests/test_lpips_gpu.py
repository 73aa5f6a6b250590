"""LPIPS (VGG) on the GPU engine (satlas_super_resolution_b200/lpips.py, metrics.calculate_lpips) against the CPU restatement of
oracle/lpips.py -- in fp32 (the metric as lpips defines it) and as a bf16 rounding model of the engine -- with seeded weights."""
import importlib.util
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore:calculate_lpips.*RANDOM:RuntimeWarning")]

SEED = 0


def fp32_bound(v):
    return 5e-3 * abs(v) + 5e-6


def bf16_bound(v):
    return 2e-3 * abs(v) + 2e-6


@pytest.fixture(autouse=True)
def _seeded_weights_only(tmp_path, monkeypatch):
    """the seeded weights of the oracle, even on a machine that holds the pretrained files"""
    monkeypatch.setenv("TORCH_HOME", str(tmp_path / "no_hub"))
    monkeypatch.chdir(tmp_path)
    for v in ("SSR_VGG16_PATH", "SSR_LPIPS_PATH", "SSR_LPIPS_RANDOM_SEED"):
        monkeypatch.delenv(v, raising=False)


def _pairs(kind, B, H, W, seed):
    """f32 [B, 3, H, W] (sr, gt) in [0, 1]-ish, as test_metrics_gpu._pairs builds them"""
    g = torch.Generator().manual_seed(seed)
    gt = torch.rand(B, 3, H, W, generator=g)
    if kind == "unrelated":
        sr = torch.rand(B, 3, H, W, generator=g)
    elif kind == "near":
        sr = gt + 0.01 * torch.randn(B, 3, H, W, generator=g)
    elif kind == "blurred":
        sr = F.avg_pool2d(gt, 5, 1, 2, count_include_pad=False)
    else:   # shifted, biased, noisy (test_metrics_gpu._pairs)
        sr = torch.roll(gt, (1, -2), (2, 3)) * 0.9 + 0.07 + 0.05 * torch.randn(B, 3, H, W, generator=g)
    return sr, gt


def _u8(kind, B, H, W, seed):
    from satlas_super_resolution_b200 import metrics as M
    sr, gt = _pairs(kind, B, H, W, seed)
    return M.to_uint8_images(sr.cuda()), M.to_uint8_images(gt.cuda())


def _oracle(a8, b8, bf16):
    from oracle import lpips as ol
    from satlas_super_resolution_b200 import weights
    vgg, lin = weights._lpips_seeded(SEED)
    return ol.lpips(a8.cpu(), b8.cpu(), vgg, lin, bf16=bf16)


def _check(got, a8, b8):
    want32, want16 = _oracle(a8, b8, False), _oracle(a8, b8, True)
    for g, w32, w16 in zip(got, want32, want16):
        assert abs(g - w32) <= fp32_bound(w32), (g, w32, w16)
        assert abs(g - w16) <= bf16_bound(w16), (g, w32, w16)
    return want32, want16


@pytest.mark.parametrize("kind", ["unrelated", "near", "blurred", "shifted"])
def test_lpips_matches_the_oracle(kind):
    from satlas_super_resolution_b200 import metrics as M
    a8, b8 = _u8(kind, 5, 128, 128, 3)
    got = M.calculate_lpips(a8, b8, lpips_model="vgg", lpips_seed=SEED)
    assert len(got) == 5 and all(isinstance(v, float) and v > 0 for v in got)
    want32, want16 = _check(got, a8, b8)
    rel32 = max(abs(g - w) / w for g, w in zip(got, want32))
    rel16 = max(abs(g - w) / w for g, w in zip(got, want16))
    print(f"lpips {kind}: values {np.round(want32, 7).tolist()}  max rel dev vs fp32 {rel32:.2e}  vs bf16 model {rel16:.2e}")


@pytest.mark.parametrize("H,W", [(256, 128), (128, 256), (144, 160)])
def test_lpips_other_sizes(H, W):
    from satlas_super_resolution_b200 import metrics as M
    a8, b8 = _u8("shifted", 2, H, W, 5)
    _check(M.calculate_lpips(a8, b8, lpips_model="vgg", lpips_seed=SEED), a8, b8)


@pytest.mark.parametrize("H,W", [(120, 120), (64, 64), (128, 120)])
def test_lpips_unsupported_sizes_raise(H, W):
    from satlas_super_resolution_b200 import metrics as M
    a8, b8 = _u8("shifted", 1, H, W, 5)
    with pytest.raises(ValueError, match="multiples of 16"):
        M.calculate_lpips(a8, b8, lpips_model="vgg", lpips_seed=SEED)


def test_lpips_identical_images_are_exactly_zero():
    from satlas_super_resolution_b200 import metrics as M
    a8, _ = _u8("unrelated", 4, 128, 128, 9)
    assert M.calculate_lpips(a8, a8.clone(), lpips_model="vgg", lpips_seed=SEED) == [0.0] * 4


def test_lpips_is_bit_reproducible_and_batch_invariant():
    from satlas_super_resolution_b200 import metrics as M
    from satlas_super_resolution_b200.ops import lib
    a8, b8 = _u8("shifted", 8, 128, 128, 11)
    first = M.calculate_lpips(a8, b8, lpips_model="vgg", lpips_seed=SEED)
    assert M.calculate_lpips(a8, b8, lpips_model="vgg", lpips_seed=SEED) == first

    def paths(fn):
        torch.cuda.synchronize()
        before = [lib().ssr_debug_conv_path_count(i) for i in range(3)]
        out = fn()
        return out, [lib().ssr_debug_conv_path_count(i) - b for i, b in zip(range(3), before)]
    _, p8 = paths(lambda: M.calculate_lpips(a8, b8, lpips_model="vgg", lpips_seed=SEED))
    for i in (0, 5):
        one, p1 = paths(lambda: M.calculate_lpips(a8[i:i + 1], b8[i:i + 1], lpips_model="vgg", lpips_seed=SEED))
        print(f"conv paths (halo, lean, streamed): batch of 8 {p8}, batch of 1 {p1}; image {i}: {first[i]!r} / {one[0]!r}")
        if p1 == p8:
            assert one[0] == first[i]
        else:
            assert abs(one[0] - first[i]) <= bf16_bound(first[i])


def test_lpips_head_is_batch_invariant_bit_for_bit():
    """the head kernels alone: a tap's value of an image does not depend on the batch around it"""
    from satlas_super_resolution_b200 import _lib as L
    from satlas_super_resolution_b200.ops import cur_stream, lib
    import ctypes as C
    g = torch.Generator().manual_seed(1)
    for Cc, h, w in ((64, 128, 128), (128, 64, 64), (512, 8, 8), (256, 8, 24)):
        B = 6
        feat = torch.relu(torch.randn(2 * B, h, w, Cc, generator=g)).to(torch.bfloat16).cuda()
        lin = (torch.rand(Cc, generator=g) * 2 / Cc).cuda()
        n = lib().ssr_lpips_cta_count(h, w)
        th, tw = (C.c_int32 * 1)(h), (C.c_int32 * 1)(w)

        def run(f, nb):
            part = torch.full((nb * n,), float("nan"), dtype=torch.float64, device="cuda")
            out = torch.empty(nb, dtype=torch.float64, device="cuda")
            L.check(lib().ssr_lpips_layer_sums(f.data_ptr(), nb, h, w, Cc, lin.data_ptr(), part.data_ptr(), cur_stream()))
            L.check(lib().ssr_lpips_finish(part.data_ptr(), nb, 1, th, tw, out.data_ptr(), cur_stream()))
            return out.cpu()
        full = run(feat, B)
        assert torch.equal(full, run(feat, B))
        i = 4
        one = run(torch.stack([feat[i], feat[B + i]]).contiguous(), 1)
        assert one[0].item() == full[i].item()
        # against the f64 head of the oracle on the same bf16 maps
        from oracle.lpips import head
        f = feat.cpu().float().permute(0, 3, 1, 2)
        want = head([f[:B]], [f[B:]], {"lin0.model.1.weight": lin.cpu().view(1, -1, 1, 1)})
        torch.testing.assert_close(full, want, rtol=2e-5, atol=1e-9)


def test_lpips_engine_is_built_once():
    from satlas_super_resolution_b200 import lpips as LP
    from satlas_super_resolution_b200 import metrics as M
    built = []
    orig = LP.LPIPSEngine.__init__

    def counting(self, *a, **k):
        built.append(1)
        orig(self, *a, **k)
    M._LPIPS_ENGINES.clear()
    LP.LPIPSEngine.__init__ = counting
    try:
        for seed in (1, 2, 3):
            a8, b8 = _u8("shifted", 2, 128, 128, seed)
            M.calculate_lpips(a8, b8, lpips_model="vgg", lpips_seed=SEED)
        eng = M.lpips_engine("cuda", SEED)
    finally:
        LP.LPIPSEngine.__init__ = orig
    assert len(built) == 1 and len(M._LPIPS_ENGINES) == 1 and list(eng._ws) == [(2, 128, 128)]


def test_validation_loop_reports_lpips_with_seeded_weights(tmp_path):
    """SSRESRGANModel.validation with psnr + lpips (lpips_model: vgg, lpips_seed: 0): the LPIPS mean over images equals the mean of
    the oracle's per-image values, and PSNR is what it is without LPIPS"""
    from oracle import metrics as om
    from satlas_super_resolution_b200 import metrics as M
    from satlas_super_resolution_b200.registry import build_model
    spec = importlib.util.spec_from_file_location("_modules_helpers", os.path.join(os.path.dirname(os.path.abspath(__file__)), "test_modules_gpu.py"))
    helpers = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(helpers)
    opt = helpers._opt(tmp_path, nb=1)
    opt["val"] = {"metrics": {"psnr": dict(type="calculate_psnr", crop_border=4, test_y_channel=False),
                              "lpips": dict(type="calculate_lpips", lpips_model="vgg", lpips_seed=SEED, better="lower")}}
    model = build_model(opt)
    loader = [helpers._batch(B=2, seed=s) for s in (11, 12)]
    assert model.validation(loader, current_iter=3, tb_logger=None, save_img=False) == 4
    psnr, l32, l16 = [], [], []
    for data in loader:
        model.feed_data(data)
        model.test()
        a8, b8 = M.to_uint8_images(model.output.float()), M.to_uint8_images(model.gt.float())
        l32 += _oracle(a8, b8, False)
        l16 += _oracle(a8, b8, True)
        for i in range(2):
            psnr.append(om.calculate_psnr(om.tensor2img(model.output[i]), om.tensor2img(model.gt[i]), 4))
    got = model.metric_results["lpips"]
    assert abs(got - float(np.mean(l32))) <= fp32_bound(np.mean(l32))
    assert abs(got - float(np.mean(l16))) <= bf16_bound(np.mean(l16))
    assert abs(model.metric_results["psnr"] - float(np.mean(psnr))) < 1e-8
    assert model.best_metric_results["val"]["lpips"]["iter"] == 3
