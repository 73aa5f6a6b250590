"""Batched validation metrics on the GPU: PSNR, SSIM (basicsr.metrics.psnr_ssim), cPSNR (ssr/metrics/cpsnr.py:7-59) and LPIPS-VGG
(ssr/metrics/lpips.py:7-21, through lpips.LPIPSEngine) for a whole batch of (SR, ground truth) pairs at once -- the reference's nondist_validation (ssr/models/ssr_esrgan_model.py:296-345) converts
one image at a time with tensor2img and runs numpy on the host (cPSNR: an 81-offset brute-force search per image).

PSNR / cPSNR: the device returns EXACT integer sums of the uint8 differences (ssr_u8_shift_diff_sums); the float64 formulas of the
reference are then evaluated on those sums.  SSIM: float64 windowed sums on the device (ssr_u8_ssim_sums).
Registered in METRIC_REGISTRY under the reference's names; `test_y_channel=True` is not built (no shipped config uses it).
"""
import math

import torch

from . import _lib as L
from .ops import cur_stream, lib
from .registry import METRIC_REGISTRY, _register


def to_uint8_images(x, rgb2bgr=True):
    """basicsr tensor2img for a batch: f32 [B, C, H, W] cuda -> uint8 [B, H, W, C] (BGR when C == 3 and rgb2bgr)"""
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 4
    x = x.contiguous()
    B, C, H, W = x.shape
    out = torch.empty((B, H, W, C), dtype=torch.uint8, device=x.device)
    L.check(lib().ssr_f32_nchw_to_u8_hwc(x.data_ptr(), out.data_ptr(), B, C, H, W, 1 if (rgb2bgr and C == 3) else 0, cur_stream()))
    return out


def _check(img, img2, test_y_channel):
    if test_y_channel:
        raise NotImplementedError("test_y_channel=True is not built on the GPU path")
    assert img.shape == img2.shape, f"Image shapes are different: {tuple(img.shape)}, {tuple(img2.shape)}."
    assert img.is_cuda and img.dtype == torch.uint8 and img.dim() == 4, "uint8 [B, H, W, C] cuda batches (to_uint8_images)"
    return img.contiguous(), img2.contiguous()


def _diff_sums(img, img2, crop_border, max_offset):
    B, H, W, C = img.shape
    n_off = (max_offset + 1) ** 2
    out = torch.zeros((B, n_off, C, 2), dtype=torch.int64, device=img.device)
    L.check(lib().ssr_u8_shift_diff_sums(img.data_ptr(), img2.data_ptr(), B, H, W, C, crop_border, max_offset, out.data_ptr(), cur_stream()))
    n = (H - 2 * crop_border - max_offset) * (W - 2 * crop_border - max_offset)
    return out.cpu(), n


def _psnr_from_mse(mse):
    return float("inf") if mse == 0 else 10.0 * math.log10(255.0 * 255.0 / mse)


def calculate_psnr(img, img2, crop_border, input_order="HWC", test_y_channel=False, **kwargs):
    """basicsr calculate_psnr over a batch -> list of floats"""
    img, img2 = _check(img, img2, test_y_channel)
    sums, n = _diff_sums(img, img2, crop_border, 0)
    C = img.shape[-1]
    return [_psnr_from_mse(int(s[0, :, 1].sum()) / (n * C)) for s in sums]


def calculate_cpsnr(img, img2, crop_border, input_order="HWC", test_y_channel=False, **kwargs):
    """ssr/metrics/cpsnr.py:7-59 over a batch: for each of the 81 relative offsets remove the per-channel brightness bias
    (mean difference) and keep the smallest MSE.  With d = img1 - img2 on the shifted crops:
    mean((d_c - mean d_c)^2 over all channels) = (sum_c S2_c - S1_c^2 / n) / (n C)."""
    img, img2 = _check(img, img2, test_y_channel)
    sums, n = _diff_sums(img, img2, crop_border, 8)
    C = img.shape[-1]
    out = []
    for s in sums:                                   # [81, C, 2]
        s1, s2 = s[:, :, 0].double(), s[:, :, 1].double()
        mse = ((s2 - s1 * s1 / n).sum(dim=1) / (n * C)).min().item()
        out.append(_psnr_from_mse(max(mse, 0.0)))
    return out


def gaussian_window_11():
    """cv2.getGaussianKernel(11, 1.5) (float64)"""
    g = [math.exp(-((i - 5) ** 2) / (2 * 1.5 * 1.5)) for i in range(11)]
    s = sum(g)
    return [v / s for v in g]


def calculate_ssim(img, img2, crop_border, input_order="HWC", test_y_channel=False, **kwargs):
    """basicsr calculate_ssim over a batch: mean over channels of the mean SSIM map (11 x 11 Gaussian window, 'valid' region)"""
    img, img2 = _check(img, img2, test_y_channel)
    B, H, W, C = img.shape
    win = torch.tensor(gaussian_window_11(), dtype=torch.float64, device=img.device)
    out = torch.zeros((B, C), dtype=torch.float64, device=img.device)
    L.check(lib().ssr_u8_ssim_sums(img.data_ptr(), img2.data_ptr(), B, H, W, C, crop_border, win.data_ptr(), out.data_ptr(), cur_stream()))
    n = (H - 2 * crop_border - 10) * (W - 2 * crop_border - 10)
    return (out / n).mean(dim=1).cpu().tolist()


def check_lpips_model(lpips_model):
    """only lpips_model 'vgg' is built (AlexNet's 11 x 11 stride-4 / 5 x 5 convs are shapes no kernel of the engine takes)"""
    if lpips_model != "vgg":
        raise NotImplementedError(f"calculate_lpips: lpips_model={lpips_model!r} is not built (only lpips_model: vgg runs on the GPU "
                                  "engine; 'alexnet' and a missing lpips_model are not supported)")


_LPIPS_ENGINES = {}      # (device, weight source) -> lpips.LPIPSEngine


def lpips_engine(device, lpips_seed=None):
    """the LPIPS engine of `device` for the weights lpips_weight_source() finds, built once and reused"""
    from . import weights
    from .lpips import LPIPSEngine
    device = torch.device(device)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    source = weights.lpips_weight_source(lpips_seed)
    key = (str(device), source)
    eng = _LPIPS_ENGINES.get(key)
    if eng is None:
        vgg, lin = weights.load_lpips_state(source)
        eng = _LPIPS_ENGINES[key] = LPIPSEngine(vgg, lin, device)
    return eng


def calculate_lpips(img, img2, lpips_model=None, lpips_seed=None, **kwargs):
    """ssr/metrics/lpips.py calculate_lpips over a batch -> list of floats: lpips.LPIPS(net='vgg') of img[i] / 255 against img2[i] / 255
    (uint8 [B, H, W, 3] cuda batches from to_uint8_images; BGR order and [0, 1] range as the reference passes them).
    lpips_seed: seeded random weights when the pretrained files are absent (tests / benchmarks)."""
    check_lpips_model(lpips_model)
    from .lpips import check_size
    assert img.shape == img2.shape, f"Image shapes are different: {tuple(img.shape)}, {tuple(img2.shape)}."
    check_size(img.shape[1], img.shape[2])
    return lpips_engine(img.device, lpips_seed).distance(img, img2)


def check_metric_opt(opt):
    """option checks that can fail before any image is processed"""
    if opt.get("type") == "calculate_lpips":
        check_lpips_model(opt.get("lpips_model"))


for _f in (calculate_psnr, calculate_ssim, calculate_cpsnr, calculate_lpips):
    _register(METRIC_REGISTRY, _f)


def calculate_metric(data, opt):
    """ssr/metrics/__init__.py:13-23 (dispatch by opt['type'])"""
    opt = dict(opt)
    return METRIC_REGISTRY.get(opt.pop("type"))(**data, **opt)
