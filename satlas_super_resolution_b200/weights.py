"""Parameter construction with the reference's state_dict key schema and init distributions.

Key schema (what published checkpoints hold, /root/reference/README.md:69-80, SURVEY.md section 5):
  G  conv_first, body.<i>.rdb<1-3>.conv<1-5>, conv_body, conv_up<1..>, conv_hr, conv_last  (.weight / .bias)
  D  conv0.{weight,bias}, conv<1-8>.{weight_orig,weight_u,weight_v}, conv9.{weight,bias}
Init (only matters for from-scratch training / benchmarks; parity tests copy weights):
  the five convs of every ResidualDenseBlock: kaiming_normal(fan_in) * 0.1, zero bias
  (/root/reference/ssr/archs/rrdbnet_arch.py:35, arch_util.py:600-628); every other conv: nn.Conv2d's default
  (uniform +-1/sqrt(fan_in) for weight and bias); spectral-norm u, v: normalised standard normal vectors.
"""
import math
from collections import OrderedDict

import torch


def _uniform(shape, bound, g):
    return (torch.rand(shape, generator=g) * 2 - 1) * bound


def rrdbnet_state(num_in_ch, num_out_ch=3, scale=4, num_feat=64, num_block=23, num_grow_ch=32, seed=0):
    g = torch.Generator().manual_seed(seed)
    if scale == 2:
        num_in_ch *= 4
    elif scale == 1:
        num_in_ch *= 16
    sd = OrderedDict()

    def plain(name, cout, cin):
        b = 1.0 / math.sqrt(cin * 9)
        sd[f"{name}.weight"] = _uniform((cout, cin, 3, 3), b, g)
        sd[f"{name}.bias"] = _uniform((cout,), b, g)

    plain("conv_first", num_feat, num_in_ch)
    for i in range(num_block):
        for j in (1, 2, 3):
            for k in range(1, 6):
                cin = num_feat + (k - 1) * num_grow_ch
                cout = num_grow_ch if k < 5 else num_feat
                sd[f"body.{i}.rdb{j}.conv{k}.weight"] = torch.randn(cout, cin, 3, 3, generator=g) * (0.1 * math.sqrt(2.0 / (cin * 9)))
                sd[f"body.{i}.rdb{j}.conv{k}.bias"] = torch.zeros(cout)
    plain("conv_body", num_feat, num_feat)
    n_up = {1: 2, 2: 2, 4: 2, 8: 3, 16: 4}[scale]
    for u in range(1, n_up + 1):
        plain(f"conv_up{u}", num_feat, num_feat)
    plain("conv_hr", num_feat, num_feat)
    plain("conv_last", num_out_ch, num_feat)
    return sd


def unet_disc_state(num_in_ch, num_feat=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    nf = num_feat
    sd = OrderedDict()
    layers = [("conv0", nf, num_in_ch, 3, True), ("conv1", 2 * nf, nf, 4, False), ("conv2", 4 * nf, 2 * nf, 4, False),
              ("conv3", 8 * nf, 4 * nf, 4, False), ("conv4", 4 * nf, 8 * nf, 3, False), ("conv5", 2 * nf, 4 * nf, 3, False),
              ("conv6", nf, 2 * nf, 3, False), ("conv7", nf, nf, 3, False), ("conv8", nf, nf, 3, False), ("conv9", 1, nf, 3, True)]
    for name, cout, cin, k, biased in layers:
        b = 1.0 / math.sqrt(cin * k * k)
        w = _uniform((cout, cin, k, k), b, g)
        if biased:
            sd[f"{name}.weight"] = w
            sd[f"{name}.bias"] = _uniform((cout,), b, g)
        else:
            sd[f"{name}.weight_orig"] = w
            u = torch.randn(cout, generator=g)
            v = torch.randn(cin * k * k, generator=g)
            sd[f"{name}.weight_u"] = u / u.norm().clamp_min(1e-12)
            sd[f"{name}.weight_v"] = v / v.norm().clamp_min(1e-12)
    return sd


VGG19_CONVS = [("conv1_1", 3, 64), ("conv1_2", 64, 64), ("conv2_1", 64, 128), ("conv2_2", 128, 128),
               ("conv3_1", 128, 256), ("conv3_2", 256, 256), ("conv3_3", 256, 256), ("conv3_4", 256, 256),
               ("conv4_1", 256, 512), ("conv4_2", 512, 512), ("conv4_3", 512, 512), ("conv4_4", 512, 512),
               ("conv5_1", 512, 512), ("conv5_2", 512, 512), ("conv5_3", 512, 512), ("conv5_4", 512, 512)]
# position of each conv inside torchvision.models.vgg19().features (for loading vgg19-dcbb9e9d.pth)
VGG19_TORCHVISION_INDEX = [0, 2, 5, 7, 10, 12, 14, 16, 19, 21, 23, 25, 28, 30, 32, 34]


def _torchvision_features(path, convs, index):
    """conv weights of a torchvision VGG checkpoint (keys features.<idx>.weight / .bias) under the conv names of `convs`"""
    raw = torch.load(path, map_location="cpu")
    sd = OrderedDict()
    for (name, _, _), idx in zip(convs, index):
        sd[f"{name}.weight"] = raw[f"features.{idx}.weight"].float()
        sd[f"{name}.bias"] = raw[f"features.{idx}.bias"].float()
    return sd


def _seeded_convs(convs, g):
    """torchvision's VGG init: kaiming_normal(fan_out, relu), zero bias"""
    sd = OrderedDict()
    for name, cin, cout in convs:
        sd[f"{name}.weight"] = torch.randn(cout, cin, 3, 3, generator=g) * math.sqrt(2.0 / (cout * 9))
        sd[f"{name}.bias"] = torch.zeros(cout)
    return sd


def vgg19_state(seed=0, pretrained_path=None):
    """VGG19 feature weights: the torchvision checkpoint when `pretrained_path` exists (keys features.<idx>.weight),
    else seeded random weights with torchvision's init (kaiming_normal fan_out, zero bias) -- the pretrained file
    cannot be downloaded offline, benchmarks and parity tests use the seeded version on both sides."""
    if pretrained_path:
        return _torchvision_features(pretrained_path, VGG19_CONVS, VGG19_TORCHVISION_INDEX)
    return _seeded_convs(VGG19_CONVS, torch.Generator().manual_seed(seed))


VGG19_FILE = "vgg19-dcbb9e9d.pth"


def vgg19_search_paths():
    """where the torchvision VGG19 checkpoint may live: $SSR_VGG19_PATH, the path basicsr looks at first (relative to the
    working directory), and the torch hub cache torchvision downloads into"""
    import os
    out = []
    if os.environ.get("SSR_VGG19_PATH"):
        out.append(os.environ["SSR_VGG19_PATH"])
    out.append(os.path.join("experiments", "pretrained_models", VGG19_FILE))
    hub = os.environ.get("TORCH_HOME") or os.path.join(os.path.expanduser("~"), ".cache", "torch")
    out.append(os.path.join(hub, "hub", "checkpoints", VGG19_FILE))
    return out


def resolve_vgg19_state(vgg_seed=None, path=None):
    """VGG19 weights for the perceptual loss.  basicsr loads the ImageNet checkpoint (downloading it when absent); a perceptual
    term on random features is meaningless for real training, so a missing checkpoint is an ERROR here unless the caller opted
    into seeded random weights explicitly (`vgg_seed` option / $SSR_VGG_RANDOM_SEED -- what tests and benchmarks use offline)."""
    import os
    import warnings
    for cand in ([path] if path else []) + vgg19_search_paths():
        if cand and os.path.exists(cand):
            return vgg19_state(pretrained_path=cand)
    if vgg_seed is None and os.environ.get("SSR_VGG_RANDOM_SEED") is not None:
        vgg_seed = int(os.environ["SSR_VGG_RANDOM_SEED"])
    if vgg_seed is None:
        raise FileNotFoundError(
            f"PerceptualLoss: {VGG19_FILE} not found (searched {vgg19_search_paths()}).  Put the torchvision VGG19 checkpoint at one "
            "of these paths or set SSR_VGG19_PATH; for tests / benchmarks without it pass vgg_seed=<int> (perceptual_opt.vgg_seed) "
            "or set SSR_VGG_RANDOM_SEED to use seeded RANDOM weights.")
    warnings.warn(f"PerceptualLoss: {VGG19_FILE} not found -- using seeded RANDOM VGG19 weights (seed {vgg_seed}); "
                  "the perceptual term is not meaningful for real training", RuntimeWarning, stacklevel=2)
    return vgg19_state(seed=vgg_seed)


# ---------------------------------------------------------------------------------------------------- LPIPS (lpips 0.1, net='vgg')
VGG16_CONVS = [("conv1_1", 3, 64), ("conv1_2", 64, 64), ("conv2_1", 64, 128), ("conv2_2", 128, 128),
               ("conv3_1", 128, 256), ("conv3_2", 256, 256), ("conv3_3", 256, 256),
               ("conv4_1", 256, 512), ("conv4_2", 512, 512), ("conv4_3", 512, 512),
               ("conv5_1", 512, 512), ("conv5_2", 512, 512), ("conv5_3", 512, 512)]
# position of each conv inside torchvision.models.vgg16().features (for loading vgg16-397923af.pth)
VGG16_TORCHVISION_INDEX = [0, 2, 5, 7, 10, 12, 14, 17, 19, 21, 24, 26, 28]
LPIPS_CHANNELS = (64, 128, 256, 512, 512)          # relu1_2, relu2_2, relu3_3, relu4_3, relu5_3
VGG16_FILE = "vgg16-397923af.pth"
LPIPS_FILE = "vgg.pth"                             # lpips/weights/v0.1/vgg.pth of the lpips package


def _lpips_seeded(seed):
    """seeded random LPIPS weights, drawn from one generator: the 13 VGG16 convs (torchvision's init), then lin0..4 as
    rand(1, C, 1, 1) * 2 / C (non-negative like the trained ones, summing to about 1 per tap)"""
    g = torch.Generator().manual_seed(seed)
    vgg = _seeded_convs(VGG16_CONVS, g)
    lin = OrderedDict((f"lin{k}.model.1.weight", torch.rand(1, c, 1, 1, generator=g) * (2.0 / c)) for k, c in enumerate(LPIPS_CHANNELS))
    return vgg, lin


def vgg16_state(seed=0, pretrained_path=None):
    """VGG16 feature weights (conv1_1 .. conv5_3): the torchvision checkpoint when `pretrained_path` is given, else the seeded ones"""
    if pretrained_path:
        return _torchvision_features(pretrained_path, VGG16_CONVS, VGG16_TORCHVISION_INDEX)
    return _lpips_seeded(seed)[0]


def lpips_lin_state(seed=0, path=None):
    """the five linear heads lin{k}.model.1.weight [1, C, 1, 1] of lpips v0.1: from the lpips weight file when `path` is given,
    else the seeded ones"""
    if path:
        raw = torch.load(path, map_location="cpu")
        return OrderedDict((f"lin{k}.model.1.weight", raw[f"lin{k}.model.1.weight"].float().reshape(1, c, 1, 1))
                           for k, c in enumerate(LPIPS_CHANNELS))
    return _lpips_seeded(seed)[1]


def _hub_dir():
    import os
    return os.path.join(os.environ.get("TORCH_HOME") or os.path.join(os.path.expanduser("~"), ".cache", "torch"), "hub", "checkpoints")


def vgg16_search_paths():
    """$SSR_VGG16_PATH, experiments/pretrained_models/ (relative to the working directory), the torch hub cache"""
    import os
    out = [os.environ["SSR_VGG16_PATH"]] if os.environ.get("SSR_VGG16_PATH") else []
    return out + [os.path.join("experiments", "pretrained_models", VGG16_FILE), os.path.join(_hub_dir(), VGG16_FILE)]


def lpips_search_paths():
    """$SSR_LPIPS_PATH, experiments/pretrained_models/, the torch hub cache, and weights/v0.1/ of an installed lpips package"""
    import importlib.util
    import os
    out = [os.environ["SSR_LPIPS_PATH"]] if os.environ.get("SSR_LPIPS_PATH") else []
    out += [os.path.join("experiments", "pretrained_models", LPIPS_FILE), os.path.join(_hub_dir(), LPIPS_FILE)]
    try:
        spec = importlib.util.find_spec("lpips")
    except (ImportError, ValueError):
        spec = None
    if spec is not None and spec.submodule_search_locations:
        out += [os.path.join(loc, "weights", "v0.1", LPIPS_FILE) for loc in spec.submodule_search_locations]
    return out


def lpips_weight_source(lpips_seed=None):
    """Which LPIPS weights to use, without loading them: ('files', vgg16 path, lin path) when both files are found, else
    ('seed', seed) when seeded random weights were asked for (`lpips_seed` option / $SSR_LPIPS_RANDOM_SEED), else
    FileNotFoundError.  An LPIPS value over random features is not the published metric, so the seeded form is opt-in only."""
    import os
    found = []
    for paths in (vgg16_search_paths(), lpips_search_paths()):
        found.append(next((p for p in paths if p and os.path.exists(p)), None))
    if all(found):
        return ("files", found[0], found[1])
    if lpips_seed is None and os.environ.get("SSR_LPIPS_RANDOM_SEED") is not None:
        lpips_seed = int(os.environ["SSR_LPIPS_RANDOM_SEED"])
    if lpips_seed is None:
        missing = [f"{name} (searched {paths})" for name, paths, f in
                   ((VGG16_FILE, vgg16_search_paths(), found[0]), (f"lpips v0.1 {LPIPS_FILE}", lpips_search_paths(), found[1])) if not f]
        raise FileNotFoundError(
            "calculate_lpips: " + "; ".join(missing) + " not found.  Put the torchvision VGG16 checkpoint and the lpips v0.1 "
            "linear-head file at one of these paths or set SSR_VGG16_PATH / SSR_LPIPS_PATH; for tests / benchmarks without them "
            "pass lpips_seed=<int> (metric option) or set SSR_LPIPS_RANDOM_SEED to use seeded RANDOM weights.")
    return ("seed", int(lpips_seed))


def load_lpips_state(source):
    """(VGG16 state, lin state) of a lpips_weight_source() result; seeded weights emit a RuntimeWarning"""
    import warnings
    if source[0] == "files":
        return vgg16_state(pretrained_path=source[1]), lpips_lin_state(path=source[2])
    warnings.warn(f"calculate_lpips: {VGG16_FILE} / lpips {LPIPS_FILE} not found -- using seeded RANDOM LPIPS weights (seed "
                  f"{source[1]}); the value is not the published LPIPS metric", RuntimeWarning, stacklevel=2)
    return _lpips_seeded(source[1])


def resolve_lpips_state(lpips_seed=None):
    """LPIPS weights under the VGG19 policy: the files when both are found, seeded random ones only on explicit request"""
    return load_lpips_state(lpips_weight_source(lpips_seed))
