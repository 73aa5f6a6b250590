"""CPU tests: the oracle (oracle/nets.py, oracle/losses.py) is pinned against
  (1) the golden fixtures produced by the UNMODIFIED reference modules (oracle/make_golden.py, oracle/make_golden_ref.py,
      tests/golden/*.pt),
  (2) the torch / torchvision / cv2 primitives the restated basicsr pieces wrap.
"""
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

import pytest
import torch
import torch.nn.functional as F

from oracle import losses, nets

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return torch.load(os.path.join(GOLD, name), map_location="cpu")


def checksum(sd):
    return float(sum(v.double().abs().sum() for v in sd.values()))


@pytest.mark.parametrize("name", ["g_small.pt", "g_full_rgb8.pt", "g_cfg1_1frame.pt", "g_12band.pt"])
def test_generator_oracle_matches_reference_golden(name):
    g = load(name)
    sd = nets.rrdbnet_init(g["num_in_ch"], 3, num_block=g["num_block"], seed=g["seed"])
    assert sum(v.numel() for v in sd.values()) == g["n_params"]
    assert abs(checksum(sd) - g["param_checksum"]) <= 1e-6 * g["param_checksum"], "seeded weights drifted"
    x = torch.rand(g["batch"], g["num_in_ch"], 32, 32, generator=torch.Generator().manual_seed(g["x_seed"]))
    with torch.no_grad():
        y = nets.rrdbnet_forward(sd, x, num_block=g["num_block"])
    assert y.shape == g["y"].shape
    assert torch.allclose(y, g["y"], atol=2e-5, rtol=1e-4), (y - g["y"]).abs().max()


def test_param_counts_match_survey():
    assert sum(v.numel() for v in nets.rrdbnet_init(24).values()) == nets.G_PARAM_COUNT_RGB8
    d = nets.unet_disc_init(27)
    n = sum(v.numel() for k, v in d.items() if not k.endswith(("weight_u", "weight_v")))
    assert n == nets.D_PARAM_COUNT_RGB8


@pytest.mark.parametrize("name", ["d_rgb8.pt", "d_plain.pt"])
def test_discriminator_oracle_matches_reference_golden(name):
    g = load(name)
    sd = nets.unet_disc_init(g["num_in_ch"], seed=g["seed"])
    assert abs(checksum(sd) - g["param_checksum"]) <= 1e-6 * g["param_checksum"]
    x = torch.rand(1, g["num_in_ch"], 64, 64, generator=torch.Generator().manual_seed(g["x_seed"]))
    p = {k: v.clone() for k, v in sd.items()}
    with torch.no_grad():
        y1 = nets.unet_disc_forward(p, x, training=True)
        y2 = nets.unet_disc_forward(p, x, training=True)
    assert torch.allclose(y1, g["y_train1"], atol=1e-5, rtol=1e-4)
    assert torch.allclose(y2, g["y_train2"], atol=1e-5, rtol=1e-4)
    for k, v in g["uv_after_2"].items():            # the power iteration advanced exactly twice
        assert torch.allclose(p[k], v, atol=1e-6), k
    with torch.no_grad():
        y3 = nets.unet_disc_forward(p, x, training=False)
    assert torch.allclose(y3, g["y_eval"], atol=1e-5, rtol=1e-4)
    # gradient through sigma (spectral-norm backward) and through the whole U-Net
    q = {k: (v.clone().requires_grad_(True) if not k.endswith(("weight_u", "weight_v")) else v.clone()) for k, v in sd.items()}
    r = torch.randn(1, 1, 64, 64, generator=torch.Generator().manual_seed(g["r_seed"]))
    (nets.unet_disc_forward(q, x, training=True) * r).sum().backward()
    assert torch.allclose(q["conv0.weight"].grad, g["grad_conv0"], atol=1e-4, rtol=1e-3)
    assert torch.allclose(q["conv3.weight_orig"].grad[:4], g["grad_conv3_head"], atol=1e-4, rtol=1e-3)
    assert abs(float(q["conv3.weight_orig"].grad.double().abs().sum()) - g["grad_conv3_abs_sum"]) < 1e-3 * g["grad_conv3_abs_sum"]


def test_pixel_unshuffle_golden():
    g = load("pixel_unshuffle.pt")
    assert torch.equal(nets.pixel_unshuffle(g["x"], 2), g["y2"])
    assert torch.equal(nets.pixel_unshuffle(g["x"], 4), g["y4"])
    assert torch.equal(nets.pixel_unshuffle(g["x"], 2), F.pixel_unshuffle(g["x"], 2))


def test_oracle_against_live_reference():
    """against what the reference's SSR_RRDBNet / SSR_UNetDiscriminatorSN produced (oracle/make_golden_ref.py, tests/golden/ref_modules.pt)"""
    g = load("ref_modules.pt")
    sd = nets.rrdbnet_init(24, 3, num_block=1, seed=g["sd_seed"])
    assert [(k, list(v.shape)) for k, v in sd.items()] == g["g1_shapes"]       # what load_state_dict(strict=True) requires
    x = torch.rand(1, 24, 32, 32, generator=torch.Generator().manual_seed(g["x_seed"]))
    with torch.no_grad():
        assert torch.allclose(g["y"], nets.rrdbnet_forward(sd, x, num_block=1), atol=1e-5)
    # the reference's own default init has the distribution oracle.nets restates
    mine = nets.rrdbnet_init(24, 3, num_block=2, seed=0)
    assert [(k, list(v.shape)) for k, v in mine.items()] == g["g2_shapes"]
    for k, std in g["g2_std"].items():
        assert abs(std / mine[k].std().item() - 1) < 0.1, k
    assert g["g2_bias_abs_max"] == 0
    dsd = nets.unet_disc_init(27, seed=7)
    assert [(k, list(v.shape)) for k, v in dsd.items()] == g["d_shapes"]


# --------------------------------------------------------------------------- restated basicsr pieces vs primitives
def test_spectral_norm_restatement_vs_torch():
    torch.manual_seed(0)
    conv = torch.nn.utils.spectral_norm(torch.nn.Conv2d(8, 16, 4, 2, 1, bias=False))
    p = {"c.weight_orig": conv.weight_orig.detach().clone(), "c.weight_u": conv.weight_u.clone(), "c.weight_v": conv.weight_v.clone()}
    x = torch.randn(2, 8, 16, 16)
    conv.train()
    for _ in range(3):
        y_ref = conv(x)
        w = nets.spectral_norm_weight(p, "c", training=True)
        assert torch.allclose(F.conv2d(x, w, None, 2, 1), y_ref, atol=1e-5)
        assert torch.allclose(p["c.weight_u"], conv.weight_u, atol=1e-6)
    conv.eval()
    assert torch.allclose(F.conv2d(x, nets.spectral_norm_weight(p, "c", training=False), None, 2, 1), conv(x), atol=1e-5)


def test_losses_vs_torch_primitives():
    g = torch.Generator().manual_seed(1)
    a, b = torch.rand(2, 3, 16, 16, generator=g), torch.rand(2, 3, 16, 16, generator=g)
    assert torch.allclose(losses.l1_loss(a, b, 0.5), 0.5 * (a - b).abs().mean())
    z = torch.randn(2, 1, 16, 16, generator=g)
    bce = torch.nn.BCEWithLogitsLoss()
    assert torch.allclose(losses.gan_loss_vanilla(z, True, is_disc=True), bce(z, torch.ones_like(z)))
    assert torch.allclose(losses.gan_loss_vanilla(z, False, is_disc=True), bce(z, torch.zeros_like(z)))
    assert torch.allclose(losses.gan_loss_vanilla(z, True, is_disc=False, loss_weight=0.1), 0.1 * bce(z, torch.ones_like(z)))
    zz = z.clone().requires_grad_(True)
    losses.gan_loss_vanilla(zz, True, is_disc=True).backward()
    assert torch.allclose(zz.grad, (torch.sigmoid(z) - 1) / z.numel(), atol=1e-7)


def test_vgg19_features_vs_torchvision():
    tv = pytest.importorskip("torchvision")
    vp = losses.vgg19_init(seed=2)
    net = tv.models.vgg19(weights=None).features.eval()
    convs = [m for m in net if isinstance(m, torch.nn.Conv2d)]
    names = [c[0] for c in losses.VGG19_LAYERS if not isinstance(c, str)]
    assert len(convs) == len(names) == 16
    with torch.no_grad():
        for m, n in zip(convs, names):
            m.weight.copy_(vp[f"{n}.weight"])
            m.bias.copy_(vp[f"{n}.bias"])
    x = torch.rand(1, 3, 64, 64, generator=torch.Generator().manual_seed(3))
    feats = losses.vgg19_features(vp, x, ["conv1_2", "conv3_4", "conv5_4"], use_input_norm=False)
    # torchvision index of the conv layers: conv1_2 = 2, conv3_4 = 16, conv5_4 = 34 (pre-ReLU outputs)
    want = {}
    t = x
    with torch.no_grad():
        for i, m in enumerate(net):
            t = m(t)
            if i in (2, 16, 34):
                want[i] = t.clone()
    assert torch.allclose(feats["conv1_2"], want[2], atol=1e-5)
    assert torch.allclose(feats["conv3_4"], want[16], atol=1e-5)
    assert torch.allclose(feats["conv5_4"], want[34], atol=1e-5)


def test_usm_sharp_pieces():
    cv2 = pytest.importorskip("cv2")
    k = losses.gaussian_kernel_1d(51, 0)
    assert abs(k.numpy() - cv2.getGaussianKernel(51, 0)[:, 0]).max() < 1e-15
    img = torch.rand(1, 3, 96, 96, generator=torch.Generator().manual_seed(4))
    kernel = torch.outer(k, k).float()
    blur = losses.filter2d(img, kernel)
    # filter2D == cv2.filter2D with BORDER_REFLECT_101 (torch 'reflect'), per plane
    ref = cv2.filter2D(img[0, 1].numpy(), -1, kernel.numpy(), borderType=cv2.BORDER_REFLECT_101)
    assert abs(blur[0, 1].numpy() - ref).max() < 1e-5
    out = losses.usm_sharp(img)
    assert out.shape == img.shape and float(out.min()) >= -1e-6 and float(out.max()) <= 1 + 1e-6
    flat = torch.full((1, 3, 96, 96), 0.5)
    assert torch.allclose(losses.usm_sharp(flat), flat, atol=1e-6)      # nothing to sharpen in a flat image


def test_metrics_oracle_against_reference_golden_and_cv2():
    """oracle/metrics.py: cPSNR equals the values the UNMODIFIED ssr/metrics/cpsnr.py produced (tests/golden/metrics_cpsnr.json,
    oracle/make_golden_metrics.py); SSIM equals basicsr's cv2.filter2D formulation; tensor2img rounds half to even like np.round."""
    import json
    import cv2
    import numpy as np
    from oracle import metrics as om
    from oracle.make_golden_metrics import image_pair
    with open(os.path.join(ROOT, "tests", "golden", "metrics_cpsnr.json")) as fh:
        gold = json.load(fh)
    for case in gold["cases"]:
        a, b = image_pair(case["seed"], c=case["channels"])
        if case.get("identical"):
            b = a.copy()
        got = om.calculate_cpsnr(a, b, case["crop_border"])
        assert got == case["cpsnr"] or abs(got - case["cpsnr"]) < 1e-12, case
    # basicsr _ssim with cv2 (the library call the restatement replaces)
    a, b = image_pair(3)
    a64, b64 = a[..., 0].astype(np.float64), b[..., 0].astype(np.float64)
    k = cv2.getGaussianKernel(11, 1.5)
    win = np.outer(k, k.transpose())
    f = lambda z: cv2.filter2D(z, -1, win)[5:-5, 5:-5]
    mu1, mu2 = f(a64), f(b64)
    c1, c2 = (0.01 * 255) ** 2, (0.03 * 255) ** 2
    ref = (((2 * mu1 * mu2 + c1) * (2 * (f(a64 * b64) - mu1 * mu2) + c2)) /
           ((mu1 ** 2 + mu2 ** 2 + c1) * ((f(a64 ** 2) - mu1 ** 2) + (f(b64 ** 2) - mu2 ** 2) + c2))).mean()
    assert abs(om._ssim(a64, b64) - ref) < 1e-10
    t = torch.tensor([[[0.5 / 255, 1.5 / 255, 2.5 / 255, -1.0, 2.0]]])          # 0.5 -> 0, 1.5 -> 2, 2.5 -> 2, clamp
    assert om.tensor2img(t).flatten().tolist() == [0, 2, 2, 0, 255]


def test_ssim_loss_restatement_properties_and_naive_evaluation():
    """oracle.losses.ssim_loss (kornia.losses.ssim_loss restated; kornia is absent offline -> "parity unpinned"): checked against a
    direct float64 evaluation of the definition (explicit reflect indexing, no conv) on a tiny image, plus ssim(x, x) = 1."""
    import math
    g = torch.Generator().manual_seed(5)
    x = torch.rand(1, 2, 6, 7, generator=g)
    y = torch.rand(1, 2, 6, 7, generator=g)
    assert abs(losses.ssim_loss(x, x).item()) < 1e-6
    k = [math.exp(-((i - 2) ** 2) / (2 * 1.5 ** 2)) for i in range(5)]
    k = [v / sum(k) for v in k]
    refl = lambda i, n: -i if i < 0 else (2 * (n - 1) - i if i >= n else i)
    tot = 0.0
    for c in range(2):
        for py in range(6):
            for px in range(7):
                m = [0.0] * 5
                for dy in range(5):
                    for dx in range(5):
                        a = x[0, c, refl(py + dy - 2, 6), refl(px + dx - 2, 7)].item()
                        b = y[0, c, refl(py + dy - 2, 6), refl(px + dx - 2, 7)].item()
                        w = k[dy] * k[dx]
                        for j, v in enumerate((a, b, a * a, b * b, a * b)):
                            m[j] += w * v
                mx, my, exx, eyy, exy = m
                num = (2 * mx * my + 1e-4) * (2 * (exy - mx * my) + 9e-4)
                den = (mx * mx + my * my + 1e-4) * ((exx - mx * mx) + (eyy - my * my) + 9e-4)
                tot += min(max((1 - num / (den + 1e-12)) / 2, 0.0), 1.0)
    assert abs(losses.ssim_loss(x, y, 0.7).item() - 0.7 * tot / (2 * 6 * 7)) < 1e-6
