"""LPIPS (lpips 0.1, net='vgg') on the engine -- the `calculate_lpips` metric of ssr/metrics/lpips.py:7-21 that the test section of
every ESRGAN config lists (esrgan_s2naip_urban.yml:181-183).

The SR and ground-truth images go through the frozen VGG16 trunk as ONE batch of 2B images (tcgen05 convs with the ReLU in the
epilogue, ssr_maxpool_relu between the blocks); the head (ssr_lpips_layer_sums per tap, ssr_lpips_finish) reduces the five post-ReLU
taps of every pair to one f64 value in a fixed order.  Forward only.  Input as calculate_lpips passes it: uint8 HWC in the BGR order
of tensor2img, scaled to [0, 1] and NOT mapped to [-1, 1] (both quirks reproduced).
"""
import ctypes as C

import torch

from . import _lib as L
from .ops import Act, PackedConv, Packer, Plan, conv_args, cur_stream, lib

VGG16_CFG = [("conv1_1", 3, 64), ("conv1_2", 64, 64), "pool1",
             ("conv2_1", 64, 128), ("conv2_2", 128, 128), "pool2",
             ("conv3_1", 128, 256), ("conv3_2", 256, 256), ("conv3_3", 256, 256), "pool3",
             ("conv4_1", 256, 512), ("conv4_2", 512, 512), ("conv4_3", 512, 512), "pool4",
             ("conv5_1", 512, 512), ("conv5_2", 512, 512), ("conv5_3", 512, 512)]
TAPS = ("conv1_2", "conv2_2", "conv3_3", "conv4_3", "conv5_3")     # relu1_2 .. relu5_3 (the stored maps are post-ReLU)
LPIPS_SHIFT = (-0.030, -0.088, -0.188)                             # lpips ScalingLayer
LPIPS_SCALE = (0.458, 0.448, 0.450)


def check_size(H, W):
    """H, W multiples of 16 (four 2 x 2 pools) and W >= 128 (the conv kernel takes maps at least 8 pixels wide: conv5 runs at W / 16)"""
    if H % 16 or W % 16 or H < 16 or W < 128:
        raise ValueError(f"calculate_lpips: image size {H} x {W} is not built -- H and W must be multiples of 16 and W >= 128 "
                         "(four 2 x 2 max pools; the conv5 block runs at W / 16 >= 8 pixels)")


class LPIPSEngine:
    def __init__(self, vgg_state, lin_state, device):
        """vgg_state: 'conv1_1.weight' / '.bias' ... (weights.vgg16_state); lin_state: 'lin{k}.model.1.weight' [1, C, 1, 1]"""
        self.device = torch.device(device)
        dev = self.device
        self.params = {k: v.to(dev, torch.float32).contiguous() for k, v in vgg_state.items()}
        self.lin = [lin_state[f"lin{k}.model.1.weight"].to(dev, torch.float32).reshape(-1).contiguous() for k in range(len(TAPS))]
        self.cv = {}
        for c in VGG16_CFG:
            if isinstance(c, str):
                continue
            name, cin, cout = c
            self.cv[name] = PackedConv(self.params[f"{name}.weight"], self.params[f"{name}.bias"], 16 if cin == 3 else cin, False, dev)
        Packer(list(self.cv.values()), dev).run()
        self.shift = torch.tensor(LPIPS_SHIFT, dtype=torch.float32, device=dev)
        self.scale = torch.tensor(LPIPS_SCALE, dtype=torch.float32, device=dev)
        self._ws = {}

    def workspace(self, B, H, W):
        key = (B, H, W)
        if key not in self._ws:
            self._ws[key] = _LWorkspace(self, B, H, W)
        return self._ws[key]

    def distance(self, img_u8, img2_u8):
        """img_u8, img2_u8: uint8 [B, H, W, 3] cuda (metrics.to_uint8_images) -> list of B floats, LPIPS(img[i], img2[i])"""
        assert img_u8.shape == img2_u8.shape, f"Image shapes are different: {tuple(img_u8.shape)}, {tuple(img2_u8.shape)}."
        assert img_u8.is_cuda and img_u8.dtype == torch.uint8 and img_u8.dim() == 4 and img_u8.shape[-1] == 3, \
            "uint8 [B, H, W, 3] cuda batches (to_uint8_images)"
        B, H, W, _ = img_u8.shape
        check_size(H, W)
        a, b = img_u8.contiguous(), img2_u8.contiguous()
        ws = self.workspace(B, H, W)
        s = cur_stream()
        lb = lib()
        for src, first in ((a, 0), (b, B)):
            L.check(lb.ssr_ingest_u8_nhwc(src.data_ptr(), B, H, W, 3, ws.inp.ptr(), 16, first, 16, self.shift.data_ptr(),
                                          self.scale.data_ptr(), s))
        ws.plan.run(s)
        return ws.out.cpu().tolist()


class _LWorkspace:
    """the 2B-image activation buffers, partial sums and the recorded launch plan of one (B, H, W)"""

    def __init__(self, eng, B, H, W):
        dev = eng.device
        lb = lib()
        B2 = 2 * B
        self.inp = Act(B2, H, W, 16, dev)
        plan = Plan()
        taps = []                       # (Act, h, w)
        cur, cur_c, hh, ww = self.inp, 16, H, W
        self._keep = [self.inp]
        for c in VGG16_CFG:
            if isinstance(c, str):
                dst = Act(B2, hh // 2, ww // 2, cur_c, dev)
                plan.add(lb.ssr_maxpool_relu, cur.ptr(), dst.ptr(), B2, hh, ww, cur_c)
                cur, hh, ww = dst, hh // 2, ww // 2
                self._keep.append(dst)
                continue
            name, _, cout = c
            pc = eng.cv[name]
            out = Act(B2, hh, ww, cout, dev)
            plan.conv(conv_args(cur.ptr(), B2, hh, ww, cur.stride, cur_c, pc.packed.data_ptr(), 3, cout, pc.n_pad,
                                bias=pc.bias.data_ptr(), act=2, out=out.ptr(), out_stride=cout))
            self._keep.append(out)
            if name in TAPS:
                taps.append((out, hh, ww))
            cur, cur_c = out, cout
        counts = [lb.ssr_lpips_cta_count(h, w) for _, h, w in taps]
        self.partial = torch.empty(B * sum(counts), dtype=torch.float64, device=dev)
        self.out = torch.empty(B, dtype=torch.float64, device=dev)
        off = 0
        for (act, h, w), lin, n in zip(taps, eng.lin, counts):
            plan.add(lb.ssr_lpips_layer_sums, act.ptr(), B, h, w, act.C, lin.data_ptr(), self.partial.data_ptr() + 8 * off)
            off += B * n
        self.tap_h = (C.c_int32 * len(taps))(*[h for _, h, _ in taps])
        self.tap_w = (C.c_int32 * len(taps))(*[w for _, _, w in taps])
        plan.add(lb.ssr_lpips_finish, self.partial.data_ptr(), B, len(taps), self.tap_h, self.tap_w, self.out.data_ptr())
        self.plan = plan
