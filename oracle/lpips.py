"""Restatement of LPIPS as ssr/metrics/lpips.py:7-21 calls it: lpips.LPIPS(net='vgg', version='0.1') in eval mode on
`torch.as_tensor(img).permute(2, 0, 1).float() / 255` of the uint8 HWC images tensor2img produced.  lpips is a requirements.txt
dependency that is not installed here -- "parity unpinned"; every piece below is cross-checked in tests/test_lpips_cpu.py against
torchvision.models.vgg16 and a hand-computed head.

  input      [0, 1] values in the BGR channel order of tensor2img, used as they are (calculate_lpips passes no normalize=True, so
             lpips sees them as if they were RGB in [-1, 1])
  scaling    (x - shift) / scale per channel, shift = [-0.030, -0.088, -0.188], scale = [0.458, 0.448, 0.450]
  trunk      torchvision vgg16().features[0:30]: 13 3 x 3 convs + ReLU, 2 x 2 max pools after conv1_2, 2_2, 3_3, 4_3
  taps       relu1_2, relu2_2, relu3_3, relu4_3, relu5_3 (C = 64, 128, 256, 512, 512)
  head       f^ = f / (sqrt(sum_c f^2) + 1e-10); d_k = sum_c lin_k[c] (f^0 - f^1)^2; value = sum_k mean_pixels(d_k)

Two modes: fp32 (the restatement) and bf16=True, a rounding model of the engine -- the scaled input, the conv weights and every
stored post-ReLU map rounded to bf16, f32 arithmetic (the engine's convs accumulate in f32, its head reads the bf16 taps).
"""
import torch
import torch.nn.functional as F

VGG16_LAYERS = [("conv1_1", 3, 64), ("conv1_2", 64, 64), "pool1",
                ("conv2_1", 64, 128), ("conv2_2", 128, 128), "pool2",
                ("conv3_1", 128, 256), ("conv3_2", 256, 256), ("conv3_3", 256, 256), "pool3",
                ("conv4_1", 256, 512), ("conv4_2", 512, 512), ("conv4_3", 512, 512), "pool4",
                ("conv5_1", 512, 512), ("conv5_2", 512, 512), ("conv5_3", 512, 512)]
TAPS = ("conv1_2", "conv2_2", "conv3_3", "conv4_3", "conv5_3")
# the torchvision vgg16().features index right after each tap's ReLU (features[:idx + 1] ends at the tap)
TAP_TORCHVISION_RELU = (3, 8, 15, 22, 29)
SHIFT = (-0.030, -0.088, -0.188)
SCALE = (0.458, 0.448, 0.450)


def _bf16(t):
    return t.to(torch.bfloat16).to(torch.float32)


def u8_to_input(img_u8):
    """uint8 [B, H, W, 3] (tensor or array) -> f32 [B, 3, H, W] in [0, 1], channel order kept (calculate_lpips' float() / 255)"""
    t = torch.as_tensor(img_u8)
    return t.permute(0, 3, 1, 2).float() / 255


def scale_input(x):
    """lpips ScalingLayer"""
    shift = torch.tensor(SHIFT, dtype=x.dtype, device=x.device).view(1, 3, 1, 1)
    scale = torch.tensor(SCALE, dtype=x.dtype, device=x.device).view(1, 3, 1, 1)
    return (x - shift) / scale


def vgg16_taps(p, x, bf16=False):
    """the five post-ReLU tap maps of the scaled input x [N, 3, H, W]; p: weights.vgg16_state names"""
    if bf16:
        x = _bf16(x)
    out = []
    for c in VGG16_LAYERS:
        if isinstance(c, str):
            x = F.max_pool2d(x, 2, 2)
            continue
        name = c[0]
        w = p[f"{name}.weight"].to(x.device, torch.float32)
        x = F.relu(F.conv2d(x, _bf16(w) if bf16 else w, p[f"{name}.bias"].to(x.device, torch.float32), padding=1))
        if bf16:
            x = _bf16(x)
        if name in TAPS:
            out.append(x)
    return out


def normalize(f, eps=1e-10):
    """lpips normalize_tensor: the eps is added to the channel norm"""
    return f / (torch.sqrt(torch.sum(f * f, dim=1, keepdim=True)) + eps)


def head(taps0, taps1, lin):
    """per-image LPIPS value (f64) from the tap lists of the two images; lin: weights.lpips_lin_state names"""
    total = 0
    for k, (f0, f1) in enumerate(zip(taps0, taps1)):
        w = lin[f"lin{k}.model.1.weight"].to(f0.device, torch.float64).view(1, -1, 1, 1)
        d = (w * (normalize(f0.double()) - normalize(f1.double())) ** 2).sum(dim=1)
        total = total + d.mean(dim=(1, 2))
    return total


def lpips(img_u8, img2_u8, vgg, lin, bf16=False):
    """uint8 [B, H, W, 3] pairs -> list of B floats"""
    x0, x1 = u8_to_input(img_u8), u8_to_input(img2_u8)
    B = x0.shape[0]
    with torch.no_grad():
        taps = vgg16_taps(vgg, scale_input(torch.cat([x0, x1])), bf16)
        return head([t[:B] for t in taps], [t[B:] for t in taps], lin).tolist()
