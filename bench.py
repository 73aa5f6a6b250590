#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on N B200s: img-pairs/s of the 8-frame ESRGAN 4x training step (configs[1]; [2] with
--gpus 8; [3] with --bands 12) and MPix/s of 16x16-chunk grid inference (configs[4], --mode infer).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--mode train|infer] [--bands 3|12] [--impl engine|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

train: a "step" = SSRESRGANModel.feed_data kernels (uint8 -> float/255, USM sharpen) + optimize_parameters
(ssr/models/ssr_esrgan_model.py:104-233: G forward, L1 + VGG19-perceptual + 0.1*GAN losses through the frozen D, G backward +
Adam + EMA, D real/fake forward+backward + Adam) on one synthetic batch of B pairs per GPU (lr uint8 [B,24|96,32,32], hr uint8
[B,3,128,128]), random-init weights (no checkpoints offline).  The model is built the way ssr/train.py builds it:
build_model(opt) -> MODEL_REGISTRY['SSRESRGANModel'].
  value : pairs/s, whole job, inputs already resident in HBM, device-timed (CUDA events, max over ranks)
  e2e   : the plugin call sequence model.feed_data({'lr','hr'} HOST pinned uint8) / model.optimize_parameters(it) /
          model.get_current_log(): H2D copy inside the timed region, loss scalars read back (D2H) every step
  roofline          : the dominant kernel, rdb_resident_kernel (a ResidualDenseBlock's five convs / five input-gradient convs per
                      launch), algorithmic FLOPs / summed device time (per-launch CUDA events in one extra eager step; with the side lane on,
                      those launches share the machine with weight-gradient / VGG launches -- `in_graph` is the kernel on its own)
  roofline_kernels  : the same for the single-launch conv kernel and the two weight-gradient kernels
  cpu_baseline      : the CPU restatement of the reference step (oracle/step.py, torch fp32) on this box's host cores
  The default run also measures the other two things BASELINE.json's metric names and attaches them to the same line:
  "infer" (grid inference MPix/s, configs[4]) and "train_12band" (configs[3] on this many GPUs) -- skip with --no-extras.
infer (--mode infer as the headline): one 2048^2 tile = 256 chunks [24,32,32] per GPU and step through infer.infer_grid
(batched forward, clamp -> uint8 -> stitch on the GPU); e2e = pinned host chunks in, uint8 canvas copied back to the host.
--impl reference: the reference's own CPU path.  The reference (pure Python on basicsr, which is not installable offline)
cannot run here, so this arm times the oracle port of it ("kind": "port") with all host threads.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# work model, BASELINE.md section 3 (FLOP = 2*MAC, convs only, per img-pair): {bands: (F_G, F_D, F_V, f_first, f_c0)}
WORK = {3: (36.7390e9, 13.4134e9, 12.7402e9, 0.0283e9, 0.5096e9), 12: (36.8239e9, 14.7723e9, 12.7402e9, 0.1132e9, 1.8686e9)}
F_RDB = 2 * 1024 * 9 * (64 * 32 + 96 * 32 + 128 * 32 + 160 * 32 + 192 * 64)      # one ResidualDenseBlock, per image: 0.4907 GFLOP
N_RDB = 69
MPIX_TILE = 2048 * 2048 / 1e6
PROFILE_CLASSES = 5   # include/ssr_b200.h: 0 conv single, 1 wgrad single, 2 chain fwd, 3 chain dgrad, 4 wgrad9 batched


def flops(bands):
    fg, fd, fv, ffirst, fc0 = WORK[bands]
    step = 3 * fg - ffirst + 8 * fd - 2 * fc0 + 3 * fv
    wgrad = fg + 2 * fd
    return dict(step=step, wgrad=wgrad, conv=step - wgrad, infer_per_chunk=fg)


def env_int(name, default):
    return int(os.environ.get(name, default))


def log(msg):
    if os.environ.get("SSR_BENCH_VERBOSE"):
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def usable_cores():
    """host threads this process may actually use: affinity mask capped by the cgroup CPU quota (os.cpu_count() reports
    the whole host, and oversubscribing a quota-limited container makes OpenMP spin for minutes)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as fq, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as fp:
                q, per = int(fq.read()), int(fp.read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel, taken from the committed `ncu --set full` capture of the same step
    (profiles/ncu_traffic.json, written by scripts/summarize_ncu.py) -- a profiler-side number, never measured in-run."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh)
    return {}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return d.get("bf16_tflops_sustained", 1379.2), d.get("bf16_tflops", 1660.0), "measured (MEASURED_PEAKS.json)"
    return 1400.0, 1590.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region: ONE nvidia-smi process looping every 200 ms
    (B200_PROFILING.md's clocks line: `-lms 200`, started before, killed after).  Spawning a fresh nvidia-smi per sample initialises
    NVML every time and holds driver locks for tens of ms -- a stall the end-to-end loop (host on the critical path every step)
    sees directly."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_flag, self.proc = index, [], False, None

    @property
    def stop_flag(self):
        return self._stop_flag

    @stop_flag.setter
    def stop_flag(self, v):
        self._stop_flag = v
        if v and self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def run(self):
        import select
        import shutil
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        base = ["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"]
        looping = False
        try:
            pre = ["stdbuf", "-oL"] if shutil.which("stdbuf") else []
            self.proc = subprocess.Popen(pre + base + ["-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
            fd, buf, t0 = self.proc.stdout.fileno(), b"", time.time()
            while not self._stop_flag:
                ready, _, _ = select.select([fd], [], [], 0.25)
                if ready:
                    chunk = os.read(fd, 65536)
                    if not chunk:
                        break
                    buf += chunk
                    *lines, buf = buf.split(b"\n")
                    for line in lines:
                        if line.strip():
                            self.rows.append([c.strip() for c in line.decode(errors="replace").split(",")])
                            looping = True
                elif not looping and time.time() - t0 > 2.0:
                    break        # nothing arrives through the pipe (block-buffered output?): one process per sample instead
        except Exception:
            pass
        finally:
            if self.proc is not None:
                try:
                    self.proc.terminate()
                except Exception:
                    pass
        while not self._stop_flag and not looping:
            try:
                out = subprocess.run(base, capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = max((int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_batch(B, seed, bands=3):
    g = torch.Generator().manual_seed(seed)
    lr = torch.randint(1, 256, (B, 8 * bands, 32, 32), generator=g, dtype=torch.uint8)
    hr = torch.randint(1, 256, (B, 3, 128, 128), generator=g, dtype=torch.uint8)
    return lr, hr


def train_config(bands):
    cin = 8 * bands
    return {"workload": f"ESRGAN 8-S2-frame {'RGB' if bands == 3 else '12-band'} training (RRDBNet-23 + UNetDiscriminatorSN, 4x), "
                        "synthetic 32x32 tiles",
            "losses": "L1(1.0) + VGG19 perceptual(conv1_2..5_4) + 0.1*GAN(vanilla), Adam 1e-4, EMA 0.999, USM gt",
            "num_in_ch_g": cin, "num_in_ch_d": cin + 3}


def model_opt(bands, graph, dist):
    """the corrected esrgan_s2naip_urban.yml (SURVEY.md section 5 / 8d: num_in_ch 24|96 and 27|99, feed_disc_lr) as build_model's opt"""
    cin = 8 * bands
    return {
        "name": "bench", "model_type": "SSRESRGANModel", "scale": 4, "num_gpu": 1, "is_train": True, "dist": dist, "manual_seed": 0,
        "l1_gt_usm": True, "percep_gt_usm": True, "gan_gt_usm": False, "feed_disc_lr": True, "cuda_graph": graph,
        "network_g": dict(type="SSR_RRDBNet", num_in_ch=cin, num_out_ch=3, num_feat=64, num_block=23, num_grow_ch=32),
        "network_d": dict(type="SSR_UNetDiscriminatorSN", num_in_ch=cin + 3, num_feat=64, skip_connection=True),
        "path": {},
        "train": {"ema_decay": 0.999,
                  "optim_g": dict(type="Adam", lr=1e-4, weight_decay=0, betas=[0.9, 0.99]),
                  "optim_d": dict(type="Adam", lr=1e-4, weight_decay=0, betas=[0.9, 0.99]),
                  "scheduler": dict(type="MultiStepLR", milestones=[400000], gamma=0.5),
                  "pixel_opt": dict(type="L1Loss", loss_weight=1.0, reduction="mean"),
                  "perceptual_opt": dict(type="PerceptualLoss", layer_weights={"conv1_2": 0.1, "conv2_2": 0.1, "conv3_4": 1, "conv4_4": 1,
                                                                                "conv5_4": 1}, vgg_type="vgg19", use_input_norm=True,
                                         perceptual_weight=1.0, style_weight=0, range_norm=False, criterion="l1",
                                         vgg_seed=2),   # seeded random VGG19: the ImageNet file cannot be fetched offline
                  "gan_opt": dict(type="GANLoss", gan_type="vanilla", real_label_val=1.0, fake_label_val=0.0, loss_weight=0.1),
                  "net_d_iters": 1, "net_d_init_iters": 0},
    }


# ---------------------------------------------------------------------------------------------- CPU arms
def cpu_step_time(batch, iters, warm, threads, bands=3):
    """the oracle restatement of the reference step (torch fp32) on the host cores; returns s/iter"""
    from oracle import losses, nets
    from oracle.step import OracleESRGAN
    torch.set_num_threads(threads)
    gp = nets.rrdbnet_init(8 * bands, 3, seed=0)
    dp = nets.unet_disc_init(8 * bands + 3, seed=1)
    vp = losses.vgg19_init(seed=2)
    orc = OracleESRGAN(gp, dp, vp, dict(ema_decay=0.999, lr=1e-4))
    lr, hr = synthetic_batch(batch, 0, bands)
    times = []
    for i in range(warm + iters):
        t0 = time.perf_counter()
        orc.feed_data(lr, hr)
        orc.optimize_parameters()
        dt = time.perf_counter() - t0
        if i >= warm:
            times.append(dt)
    return sum(times) / len(times)


def cpu_infer_time(chunks, iters, warm, threads):
    """the reference generator forward (oracle/nets.py = rrdbnet_arch.py:116-137) on `chunks` 32x32 chunks under no_grad; s/iter"""
    from oracle import nets
    torch.set_num_threads(threads)
    gp = nets.rrdbnet_init(24, 3, seed=0)
    x = synthetic_batch(chunks, 0)[0].float() / 255
    times = []
    with torch.no_grad():
        for i in range(warm + iters):
            t0 = time.perf_counter()
            out = nets.rrdbnet_forward(gp, x)
            (out.clamp(0, 1) * 255).to(torch.uint8)
            dt = time.perf_counter() - t0
            if i >= warm:
                times.append(dt)
    return sum(times) / len(times)


CPU_TRAIN_BATCH = 8     # BASELINE.md section 4: 8-frame full step, B = 8 (CPU throughput is flat in B)
CPU_INFER_CHUNKS = 16   # BASELINE.md section 4 (4): G forward under no_grad, B = 16 chunks


def cpu_baseline(mode, bands, steps, warm):
    threads = usable_cores()
    if mode == "infer":
        t = cpu_infer_time(CPU_INFER_CHUNKS, steps, warm, threads)
        val = CPU_INFER_CHUNKS * 128 * 128 / 1e6 / t
        return dict(value=val, unit="MPix/s", cores=threads, kind="port", t=t, steps=steps, batch=CPU_INFER_CHUNKS,
                    sample=f"{steps} timed generator forwards of {CPU_INFER_CHUNKS} chunks [24,32,32] (oracle/nets.py, torch fp32 CPU, all host "
                           f"threads) after {warm} warm-up")
    t = cpu_step_time(CPU_TRAIN_BATCH, steps, warm, threads, bands)
    return dict(value=CPU_TRAIN_BATCH / t, unit="img-pairs/s", cores=threads, kind="port", t=t, steps=steps, batch=CPU_TRAIN_BATCH,
                sample=f"{steps} timed optimize_parameters steps of {CPU_TRAIN_BATCH} pairs (oracle/step.py, torch fp32 CPU, all host threads) "
                       f"after {warm} warm-up; the reference itself needs basicsr, which is absent offline")


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    cb = cpu_baseline(args.mode, args.bands, steps, warm)
    t = cb.pop("t")
    cb.pop("steps")
    batch = cb.pop("batch")
    metric = "infer MPix/s (16x16-chunk grid inference, 8-frame RRDBNet-23)" if args.mode == "infer" else "img-pairs/sec 8-frame ESRGAN 4x train"
    cfg = dict(workload="ssr/infer_grid.py 16x16-chunk stitched inference, 8-frame model") if args.mode == "infer" else train_config(args.bands)
    line = {"impl": "reference", "metric": metric, "value": cb["value"], "unit": cb["unit"],
            "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": t * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(cfg, batch_per_step=batch),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": cb["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------- engine arm
class Harness:
    def __init__(self, world):
        self.world = world

    def barrier(self):
        torch.cuda.synchronize()
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, k):
        """k calls of fn between barrier + synchronize on both sides, device-timed, max over ranks -> total ms"""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if self.world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return ms.item()


def dump_outputs(path, arrays):
    """--dump-outputs: each array as <path>/<name>.npy in float32 (float64 for loss scalars), so two builds can be compared"""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        np.save(os.path.join(path, f"{name}.npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def train_state(tr):
    """every tensor a training step reads and updates: parameters, spectral-norm vectors, EMA copy, Adam moments (the packed
    weights are rebuilt from these at the start of each step)"""
    return tr.replicated_tensors() + [t for o in (tr.opt_g, tr.opt_d) for t in (o.m.flat, o.v.flat)]


def restore_train_state(tr, saved):
    for t, s in zip(train_state(tr), saved):
        t.copy_(s)
    for o in (tr.opt_g, tr.opt_d):
        o.step_count = 0
        o.sync_device_hyper()


def train_outputs(model):
    """what a caller of optimize_parameters receives after the step: the generator output and the loss scalars.  The updated
    weights are optimizer state, not an output, and are left out: one Adam step from zero moments moves every weight by
    lr * sign(gradient), so a gradient element at the rounding level of the atomic reductions flips by 2 * lr."""
    out = {"output": model.output.float()}
    out.update({k: torch.tensor(v, dtype=torch.float64) for k, v in model.get_current_log().items()})
    return out


def roofline_entry(kernel, flop, ms, count, peak, peak_src, extra=None):
    ach = flop / (ms / 1e3) / 1e12 if ms > 0 else None
    d = {"kernel": kernel, "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak if ach else None,
         "peak_source": peak_src, "launches_per_step": int(count), "ms_per_step": ms,
         "flop_per_launch": flop / max(1, count), "us_per_launch": ms * 1e3 / max(1, count)}
    if extra:
        d.update(extra)
    return d


def measure_train(args, bands, rank, world, local, lib, L, harness, steps, warmup, dump=None):
    from satlas_super_resolution_b200.ops import cur_stream
    from satlas_super_resolution_b200.registry import build_model
    B = args.batch
    torch.manual_seed(rank)            # ssr/utils/options.py:81 seeds every rank with manual_seed + rank; rank 0's init is broadcast
    model = build_model(model_opt(bands, not args.no_graph, world > 1))
    tr = model.trainer
    initial = [t.clone() for t in train_state(tr)]
    lr_h, hr_h = synthetic_batch(B, rank, bands)
    data = {"lr": lr_h.pin_memory(), "hr": hr_h.pin_memory()}
    it = [0]

    def step_resident():
        it[0] += 1
        tr._feed_kernels(tr.io, cur_stream())
        model.optimize_parameters(it[0])

    def step_e2e():
        it[0] += 1
        model.feed_data(data)
        model.optimize_parameters(it[0])
        return model.get_current_log()

    log(f"model built ({bands} bands)")
    model.feed_data(data)
    for i in range(warmup):
        step_resident()
        torch.cuda.synchronize()
        log(f"warm-up step {i} done")
    # The last timed step starts again from the seeded initial state (restored between two timed spans): the weight and
    # spectral-norm reductions sum with f32 atomics in no fixed order, and the GAN game amplifies those last-bit differences
    # step by step, so only a step from a fixed state computes the same outputs in every run.  A step's work does not depend
    # on the weight values.
    ms_total = harness.timed(step_resident, steps - 1) if steps > 1 else 0.0
    restore_train_state(tr, initial)
    del initial
    ms_total += harness.timed(step_resident, 1)
    log(f"resident timing done: {ms_total / steps:.2f} ms/step")
    if dump:
        outs = train_outputs(model)           # every rank: the loss read-back reduces over ranks
        if rank == 0:
            dump_outputs(dump, outs)
    # The end-to-end loop has the host on the critical path every step (H2D, graph launch, loss read-back): ONE stall of the host thread
    # (another process holding a driver lock for tens of ms) shifts a 20-step average by several per cent -- one run of the pool showed
    # 24 instead of 16.7 ms.  Two K-step passes; the faster one is reported, both are listed in the line (e2e.passes_ms_per_step).
    e2e_passes = [harness.timed(step_e2e, steps) for _ in range(2)]
    ms_e2e = min(e2e_passes)
    log(f"e2e timing done: {ms_e2e / steps:.2f} ms/step (passes: {[round(p / steps, 3) for p in e2e_passes]})")
    # ---- one eager, instrumented step: per-launch CUDA events around the tensor-core kernels (graph replays do not pass
    # through the host entry points, so launches are also counted here)
    tr.use_graph = False
    tr._warm.clear()
    L.check(lib.ssr_profile_start())
    l0 = lib.ssr_launch_count()
    step_resident()
    launches = lib.ssr_launch_count() - l0
    ms_cls = (ctypes.c_double * PROFILE_CLASSES)()
    cnt_cls = (ctypes.c_int64 * PROFILE_CLASSES)()
    L.check(lib.ssr_profile_stop(ms_cls, cnt_cls, PROFILE_CLASSES))
    tr.use_graph = not args.no_graph
    # ---- the dense-block launches as they run inside the step's graph: back to back with programmatic dependent launch (the
    # per-launch events above sit BETWEEN the launches and forbid that overlap: +6 .. 8 us per launch).  The 69 forward launches
    # of the generator's own forward plan / the 69 input-gradient launches of its backward plan, same buffers, one graph each.
    graph_us = {}
    try:
        from satlas_super_resolution_b200.ops import Plan
        h, w = lr_h.shape[-2] // tr.G.unshuffle, lr_h.shape[-1] // tr.G.unshuffle
        ws = tr.G.workspace(B, h, w, True)
        for key, plan, fn in (("forward", ws.fwd, lib.ssr_conv_tc_chain), ("input_gradient", ws.bwd, lib.ssr_conv_tc_chain_acc)):
            calls = [c for c in (plan.calls if plan is not None else []) if c[0] is fn or getattr(c[0], "__name__", "") == fn.__name__]
            if not calls:
                continue
            sub = Plan()
            sub.calls = calls
            side = torch.cuda.Stream()
            with torch.cuda.stream(side):
                sub.run(cur_stream())
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side):
                    sub.run(cur_stream())
                for _ in range(2):
                    g.replay()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(5):
                    g.replay()
                e1.record()
                torch.cuda.synchronize()
            graph_us[key] = {"launches": len(calls), "us_per_launch": e0.elapsed_time(e1) * 1e3 / (5 * len(calls))}
    except Exception as exc:   # diagnostics only: the per-launch numbers above stand on their own
        log(f"back-to-back dense-block timing skipped: {exc!r}")
    return dict(B=B, ms_step=ms_total / steps, ms_e2e=ms_e2e / steps, launches=int(launches), ms_cls=list(ms_cls), cnt_cls=list(cnt_cls),
                h2d=int(lr_h.numel() + hr_h.numel()), model=model, graph_us=graph_us, side_lane=bool(getattr(tr, "overlap", False)),
                e2e_passes=[p / steps for p in e2e_passes])


def train_rooflines(m, bands, peak, peak_src):
    f = flops(bands)
    B = m["B"]
    ms, cnt = m["ms_cls"], m["cnt_cls"]
    chain_flop = N_RDB * F_RDB * B
    traffic = ncu_traffic()
    t_chain = dict(traffic.get("rdb_resident_kernel") or traffic.get("conv_chain_kernel") or {})
    main = roofline_entry("ssr::rdb_resident_kernel (ResidualDenseBlocks -- up to twelve, four RRDBs, per launch: their five forward convs each, or their five "
                          "input-gradient convs; tcgen05 implicit GEMM over a shared-memory-resident 192-channel tile, one 4-CTA cluster per image)", 2 * chain_flop, ms[2] + ms[3], cnt[2] + cnt[3], peak, peak_src,
                          dict(traffic=t_chain.get("dram_bytes_per_launch"), traffic_note=t_chain.get("note"),
                               forward=roofline_entry("rdb_resident_kernel<false>, forward", chain_flop, ms[2], cnt[2], peak, peak_src),
                               input_gradient=roofline_entry("rdb_resident_kernel<true>, input gradient", chain_flop, ms[3], cnt[3], peak, peak_src)))
    # in-graph figure: the same launches back to back in a CUDA graph (what the step replays); operand ceiling: an SS-form
    # tcgen05.mma M = 128, N, K = 16 reads (4096 + 32 N) B of shared memory at 128 B / clk = 32 + N / 4 cycles for N / 2 cycles of math
    gu = m.get("graph_us") or {}
    if gu:
        per_block_flop = chain_flop / N_RDB
        for key, ent in gu.items():
            # one launch takes ssr_rdb_resident_max_blocks consecutive blocks (four RRDBs): report per launch AND per dense block
            us_block = ent["us_per_launch"] * ent["launches"] / N_RDB
            ent["us_per_block"] = us_block
            ach = per_block_flop / (us_block * 1e-6) / 1e12
            main[key]["in_graph"] = {"us_per_launch": ent["us_per_launch"], "us_per_block": us_block, "blocks_per_launch": N_RDB / ent["launches"],
                                     "achieved": ach, "frac": ach / peak, "launches": ent["launches"],
                                     "how": "the generator's own dense-block launches of one pass, captured back to back in one CUDA graph (programmatic dependent launch active), CUDA events around 5 replays"}
        if "forward" in gu and "input_gradient" in gu:
            us = 0.5 * (gu["forward"]["us_per_block"] + gu["input_gradient"]["us_per_block"])
            ach = per_block_flop / (us * 1e-6) / 1e12
            main["in_graph"] = {"us_per_block": us, "achieved": ach, "frac": ach / peak}
    main["timing"] = ("per-launch CUDA events (on the launching stream) in one eager step" +
                      (" WITH the side lane: the input-gradient launches share the machine with the previous group's weight-gradient launches, the "
                       "forward launches with the ground-truth VGG pass (the kernel on its own: in_graph)" if m.get("side_lane") else ""))
    main["operand_ceiling"] = {"forward_frac_of_peak": (504 * 16 + 216 * 32) / (504 * 40 + 216 * 48),
                               "note": "shared-memory operand bandwidth of SS-form MMAs: the forward block issues 504 MMAs with N = 32 (16 cycles of math, 40 of operand reads) and 216 with N = 64 (32 / 48); profiles/r02_conv64_ncu.md"}
    others = {
        "conv_tc_kernel": roofline_entry("ssr::conv_tc_kernel (single-launch convs: G head / tail, D, VGG19; forward + input gradient)",
                                         f["conv"] * B - 2 * chain_flop, ms[0], cnt[0], peak, peak_src),
        "wgrad9_tc_batched_kernel": roofline_entry("ssr::wgrad9_tc_batched_kernel (five weight gradients of a dense block per launch)",
                                                   chain_flop, ms[4], cnt[4], peak, peak_src),
        "wgrad_tc_kernels": roofline_entry("ssr::wgrad9_tc_kernel / wgrad_tc_kernel (weight gradients outside the trunk)",
                                           f["wgrad"] * B - chain_flop, ms[1], cnt[1], peak, peak_src),
        "all_conv_fwd_dgrad": roofline_entry("every forward / input-gradient conv", f["conv"] * B, ms[0] + ms[2] + ms[3], cnt[0] + cnt[2] + cnt[3],
                                             peak, peak_src),
    }
    return main, others


def measure_infer(args, rank, world, harness, steps, warmup, dump=None):
    from satlas_super_resolution_b200 import weights
    from satlas_super_resolution_b200.archs import SSR_RRDBNet
    from satlas_super_resolution_b200.infer import infer_grid
    net = SSR_RRDBNet(24, 3)
    net.load_state_dict(weights.rrdbnet_state(24, 3, seed=0))
    net = net.cuda().eval()
    # weak scaling: every rank stitches its own tile (tiles are independent -- replicas, no collective: ssr/infer_grid.py:46-85)
    lr_h = synthetic_batch(256, 1000 + rank)[0].pin_memory()
    lr_d = lr_h.cuda()
    host_canvas = torch.empty((2048, 2048, 3), dtype=torch.uint8).pin_memory()
    last = [None]

    def step_resident():
        last[0] = infer_grid(net, lr_d, batch=args.infer_batch)

    def step_e2e():
        host_canvas.copy_(infer_grid(net, lr_h, batch=args.infer_batch), non_blocking=True)

    for _ in range(warmup):
        step_resident()
    ms = harness.timed(step_resident, steps) / steps
    if dump and rank == 0:
        dump_outputs(dump, {"canvas": last[0]})      # the stitched uint8 [2048, 2048, 3] tile, 48 MiB as float32
    last[0] = None
    for _ in range(2):
        step_e2e()
    ms_e2e = harness.timed(step_e2e, steps) / steps
    from satlas_super_resolution_b200 import _lib as L
    lib = L.load()
    l0 = lib.ssr_launch_count()
    step_resident()
    torch.cuda.synchronize()
    return dict(ms_step=ms, ms_e2e=ms_e2e, launches=int(lib.ssr_launch_count() - l0), h2d=int(lr_h.numel()), d2h=int(host_canvas.numel()))


def infer_block(m, world, peak, peak_src, steps, warmup):
    f = flops(3)
    val = world * MPIX_TILE / (m["ms_step"] / 1e3)
    tflops = 256 * f["infer_per_chunk"] / (m["ms_step"] / 1e3) / 1e12
    return {"metric": "infer MPix/s (16x16-chunk grid inference, 8-frame RRDBNet-23)", "value": val, "unit": "MPix/s",
            "ms_per_step": m["ms_step"], "steps": steps, "warmup": warmup,
            "config": {"workload": "ssr/infer_grid.py: one 2048^2 tile (256 chunks [24,32,32] -> 128x128, stitched) per GPU and step",
                       "chunks_per_gpu_per_step": 256, "parallelism": f"replicas x{world} (independent tiles, no collective)"},
            "e2e": {"value": world * MPIX_TILE / (m["ms_e2e"] / 1e3), "unit": "MPix/s", "h2d_bytes_per_step": m["h2d"],
                    "d2h_bytes_per_step": m["d2h"]},
            "gpu_launches_per_step": m["launches"],
            "roofline": {"kernel": "generator forward (conv_chain_kernel + conv_tc_kernel)", "bound": "tensor", "achieved": tflops, "peak": peak,
                         "unit": "TFLOP/s", "frac": tflops / peak, "peak_source": peak_src,
                         "flop_per_step": 256 * f["infer_per_chunk"], "note": "2.2424 TFLOP per output MPix (BASELINE.md section 3)"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=32, help="pairs per GPU per step (reference batch_size_per_gpu: 32)")
    ap.add_argument("--mode", default="train", choices=["train", "infer"])
    ap.add_argument("--bands", type=int, default=3, choices=[3, 12], help="3 = RGB (24-channel G input), 12 = all Sentinel-2 bands (96)")
    ap.add_argument("--infer-batch", type=int, default=256, help="chunks per generator forward in --mode infer")
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="train mode: skip the attached inference / 12-band measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the headline measurement computed in its last timed step to "
                                                          "DIR/<name>.npy (rank 0), for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl engine")
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))

    from satlas_super_resolution_b200 import _lib as L
    lib = L.load()
    harness = Harness(world)
    peak_sus, peak_burst, peak_src = measured_peaks()
    peak_note = f"{peak_src}: bf16_tflops_sustained (kernels timed inside a long step)"
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    if args.mode == "infer":
        m = measure_infer(args, rank, world, harness, args.steps, args.warmup, args.dump_outputs)
        sampler.stop_flag = True
        if rank == 0:
            blk = infer_block(m, world, peak_sus, peak_note, args.steps, args.warmup)
            line = {"metric": blk["metric"], "value": blk["value"], "unit": "MPix/s", "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": m["ms_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                    "dtype": "bf16", "data": "synthetic",
                    "config": dict(blk["config"], l2="256 chunks stream ~0.9 GB of activations per step, far above the 126 MB L2"),
                    "e2e": blk["e2e"], "gpu_launches": m["launches"] * args.steps, "gpu_launches_per_step": m["launches"],
                    "roofline": blk["roofline"], "clocks": sampler.summary()}
            if not args.no_cpu_baseline:
                cb = cpu_baseline("infer", 3, 2, 1)
                for k in ("t", "steps", "batch"):
                    cb.pop(k)
                line["cpu_baseline"] = cb
            print(json.dumps(line), flush=True)
        if world > 1:
            torch.distributed.destroy_process_group()
        return

    bands = args.bands
    m = measure_train(args, bands, rank, world, local, lib, L, harness, args.steps, args.warmup, args.dump_outputs)
    sampler.stop_flag = True
    clocks = sampler.summary() if rank == 0 else None
    extras = {}
    if not args.no_extras:
        # the other two halves of BASELINE.json's metric, measured in the same run
        k, w = args.steps, args.warmup
        del m["model"]
        torch.cuda.empty_cache()
        mi = measure_infer(args, rank, world, harness, k, w)
        if rank == 0:
            extras["infer"] = infer_block(mi, world, peak_sus, peak_note, k, w)
        other = 12 if bands == 3 else 3
        mo = measure_train(args, other, rank, world, local, lib, L, harness, k, w)
        if rank == 0:
            fo = flops(other)
            main_o, _ = train_rooflines(mo, other, peak_sus, peak_note)
            extras["train_12band" if other == 12 else "train_rgb"] = {
                "metric": "img-pairs/sec 8-frame ESRGAN 4x train", "value": mo["B"] * world / (mo["ms_step"] / 1e3), "unit": "img-pairs/s",
                "ms_per_step": mo["ms_step"], "steps": k, "warmup": w, "config": dict(train_config(other), batch_per_gpu=mo["B"]),
                "e2e": {"value": mo["B"] * world / (mo["ms_e2e"] / 1e3), "unit": "img-pairs/s", "h2d_bytes_per_step": mo["h2d"],
                        "d2h_bytes_per_step": 32},
                "step_tflops": fo["step"] * mo["B"] / (mo["ms_step"] / 1e3) / 1e12, "gpu_launches_per_step": mo["launches"],
                "roofline": main_o}
        del mo
    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    f = flops(bands)
    B = m["B"]
    value = B * world / (m["ms_step"] / 1e3)
    main_r, other_r = train_rooflines(m, bands, peak_sus, peak_note)
    line = {
        "metric": "img-pairs/sec 8-frame ESRGAN 4x train", "value": value, "unit": "img-pairs/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["ms_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": dict(train_config(bands), batch_per_gpu=B, global_batch=B * world, parallelism=f"dp{world}",
                       cuda_graph=not args.no_graph, side_lane=m.get("side_lane", False), api="build_model(opt) -> SSRESRGANModel.feed_data / optimize_parameters / get_current_log",
                       l2="no explicit flush: one step streams >10 GB of activations/gradients, far above the 126 MB L2"),
        "e2e": {"value": B * world / (m["ms_e2e"] / 1e3), "unit": "img-pairs/s", "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": 32,
                "passes_ms_per_step": m.get("e2e_passes"), "how": f"the faster of two {args.steps}-step passes (the host is on the critical path every step)"},
        "gpu_launches": m["launches"] * args.steps, "gpu_launches_per_step": m["launches"],
        "step_flop_fraction_of_peak": f["step"] * B / (m["ms_step"] / 1e3) / 1e12 / peak_sus,
        "step_tflops": f["step"] * B / (m["ms_step"] / 1e3) / 1e12,
        "roofline": main_r, "roofline_kernels": other_r, "clocks": clocks,
    }
    line.update(extras)
    if not args.no_cpu_baseline:
        log(f"cpu baseline on {usable_cores()} threads")
        cb = cpu_baseline("train", bands, 2, 1)
        for k in ("t", "steps", "batch"):
            cb.pop(k)
        line["cpu_baseline"] = cb
    print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
