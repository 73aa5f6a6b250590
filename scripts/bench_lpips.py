"""LPIPS-VGG throughput: image pairs/s at 128 x 128 for B = 1, 16, 256 (CUDA events, warm-up first), the engine's
metrics.calculate_lpips against three baselines on the same GPU:
  torch_tf32     the same computation (oracle/lpips.py restatement, f32 head like lpips) through stock PyTorch / cuDNN in fp32 with
                 TF32 convolutions -- the arithmetic of lpips.LPIPS on a GPU with torch's defaults
  torch_bf16     the same under torch.autocast(bfloat16)
  ref_loop       the reference's per-image loop (ssr/metrics/lpips.py: host HWC uint8 -> cuda -> float / 255 -> LPIPS -> .item()), with
                 the network built once instead of once per image
Seeded weights (the pretrained files are not needed for timing).  Every call of every variant returns host floats.
Usage: python scripts/bench_lpips.py [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys
import warnings

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import lpips as ol  # noqa: E402
from satlas_super_resolution_b200 import metrics as M  # noqa: E402
from satlas_super_resolution_b200 import weights  # noqa: E402

H = W = 128
REPS = {1: 100, 16: 30, 256: 6}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"nvidia-smi unavailable: {e}"
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def torch_lpips(vgg, lin, x0, x1):
    """lpips.LPIPS(net='vgg') forward on [0, 1] inputs as calculate_lpips passes them, in torch ops (f32 head)"""
    taps = ol.vgg16_taps(vgg, ol.scale_input(torch.cat([x0, x1])))
    B = x0.shape[0]
    val = 0
    for k, t in enumerate(taps):
        t = t.float()
        e = (ol.normalize(t[:B]) - ol.normalize(t[B:])) ** 2
        val = val + F.conv2d(e, lin[f"lin{k}.model.1.weight"]).mean(dim=(2, 3))
    return val.view(-1)


def timed(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_lpips needs a GPU"
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    warnings.simplefilter("ignore", RuntimeWarning)
    vgg, lin = weights._lpips_seeded(0)
    vgg_d = {k: v.cuda() for k, v in vgg.items()}
    lin_d = {k: v.cuda() for k, v in lin.items()}
    res = {"metric": "LPIPS-VGG image pairs/s at 128x128 (higher is better)", "card": card(), "rows": []}
    g = torch.Generator().manual_seed(0)
    for B in (1, 16, 256):
        sr = torch.rand(B, 3, H, W, generator=g)
        gt = (sr + 0.05 * torch.randn(B, 3, H, W, generator=g))
        a8, b8 = M.to_uint8_images(sr.cuda()), M.to_uint8_images(gt.cuda())
        a_host, b_host = a8.cpu().numpy(), b8.cpu().numpy()
        x0, x1 = ol.u8_to_input(a8), ol.u8_to_input(b8)
        eng_vals = M.calculate_lpips(a8, b8, lpips_model="vgg", lpips_seed=0)
        row = {"B": B, "engine_values_head": eng_vals[:2]}

        def engine():
            return M.calculate_lpips(a8, b8, lpips_model="vgg", lpips_seed=0)

        def t_tf32():
            with torch.no_grad():
                return torch_lpips(vgg_d, lin_d, ol.u8_to_input(a8), ol.u8_to_input(b8)).tolist()

        def t_bf16():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                return torch_lpips(vgg_d, lin_d, ol.u8_to_input(a8), ol.u8_to_input(b8)).tolist()

        def ref_loop():
            out = []
            with torch.no_grad():
                for i in range(B):
                    t1 = torch.as_tensor(a_host[i]).permute(2, 0, 1).unsqueeze(0).cuda().float() / 255
                    t2 = torch.as_tensor(b_host[i]).permute(2, 0, 1).unsqueeze(0).cuda().float() / 255
                    out.append(torch_lpips(vgg_d, lin_d, t1, t2).item())
            return out
        for name, fn in (("engine", engine), ("torch_tf32", t_tf32), ("torch_bf16", t_bf16), ("ref_loop", ref_loop)):
            reps = REPS[B] if name != "ref_loop" else max(2, REPS[B] // max(1, B // 16))
            ms = timed(fn, reps)
            vals = fn()
            dev = max(abs(v - e) / max(abs(e), 1e-12) for v, e in zip(vals, eng_vals))
            row[name] = {"ms_per_call": round(ms, 4), "pairs_per_s": round(B / (ms / 1e3), 1), "reps": reps,
                         "max_rel_diff_vs_engine": float(f"{dev:.3e}")}
        for name in ("torch_tf32", "torch_bf16", "ref_loop"):
            row[f"speedup_vs_{name}"] = round(row[name]["ms_per_call"] / row["engine"]["ms_per_call"], 2)
        res["rows"].append(row)
        print(json.dumps(row), flush=True)
    res["card_after"] = card()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
