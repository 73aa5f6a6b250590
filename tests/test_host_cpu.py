"""CPU tests (no GPU): the C-ABI library loads and exports every symbol include/ssr_b200.h declares, compute entry points
fail loudly without a device, host-side helpers (flat buffers, sharding, cgroup-aware core count) and the world_size-2
gloo path of the gradient exchange."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    with open(os.path.join(ROOT, "include", "ssr_b200.h")) as fh:
        return sorted(set(re.findall(r"\b(ssr_[a-z0-9_]+)\s*\(", fh.read())))


def test_library_builds_loads_and_exports_the_header():
    from satlas_super_resolution_b200 import _lib, _protos
    lib = _lib.load()
    names = header_symbols()
    assert len(names) >= 35
    for n in names:
        assert hasattr(lib, n), f"libssr_b200.so does not export {n}"
    bound = set(_protos.PROTOS) | {"ssr_last_error", "ssr_abi_version", "ssr_launch_count", "ssr_conv_tc", "ssr_conv_tc_chain", "ssr_conv_tc_chain_acc",
                                   "ssr_conv_tc_chain_acc_supported", "ssr_rdb_resident_max_blocks",
                                   "ssr_packed_weight_bytes", "ssr_pack_conv_weight"}
    assert set(names) <= bound, f"no ctypes prototype for {set(names) - bound}"
    assert lib.ssr_abi_version() == 1
    # struct mirrors have the C sizes (checked against static_asserts in the library for the device-side tables)
    assert C.sizeof(_protos.PackDesc) == 48 and C.sizeof(_protos.SnDesc) == 64 and C.sizeof(_protos.UnpackDesc) == 48


@pytest.mark.skipif(torch.cuda.is_available(), reason="this checks the no-GPU behaviour")
def test_compute_calls_fail_loudly_without_a_gpu():
    from satlas_super_resolution_b200 import _lib
    lib = _lib.load()
    a = _lib.ConvTcArgs()
    a.r, a.n_img, a.h, a.w, a.cin, a.x_pix_stride, a.cout, a.n_pad = 3, 1, 32, 32, 64, 64, 32, 32
    buf = (C.c_char * 4096)()
    a.x = C.addressof(buf) // 128 * 128 + 128
    a.w_packed = a.x
    rc = lib.ssr_conv_tc(C.byref(a), None)
    assert rc == -2, "a compute call without a CUDA device must return SSR_E_CUDA, not fall back"
    assert lib.ssr_last_error()
    with pytest.raises(_lib.SsrError):
        _lib.check(rc)


def test_flat_buffer_and_sharding():
    from collections import OrderedDict
    from satlas_super_resolution_b200.ops import FlatBuffer, rank_slice
    fb = FlatBuffer(OrderedDict(a=(3, 5), b=(7,), c=(2, 2, 2)), "cpu")
    assert fb.numel == 3 * 64 and all(off % 64 == 0 for off, _, _ in fb.offsets.values())
    fb.view("b").fill_(2.0)
    assert fb.flat.sum() == 14 and fb.view("a").shape == (3, 5)
    g = fb.like()
    assert g.offsets is fb.offsets and g.flat.abs().sum() == 0
    items = [list(rank_slice(256, r, 8)) for r in range(8)]
    assert sorted(sum(items, [])) == list(range(256)) and all(len(i) == 32 for i in items)
    assert [len(rank_slice(10, r, 4)) for r in range(4)] == [3, 3, 3, 1]


def test_bench_helpers():
    sys.path.insert(0, ROOT)
    import bench
    n = bench.usable_cores()
    assert 1 <= n <= (os.cpu_count() or 1)
    a, _ = bench.synthetic_batch(2, 0)
    b, _ = bench.synthetic_batch(2, 1)
    assert a.dtype == torch.uint8 and a.min() >= 1 and not torch.equal(a, b)
    f3, f12 = bench.flops(3), bench.flops(12)
    assert abs(f3["step"] / 1e9 - 254.70) < 0.01 and abs(f12["step"] / 1e9 - 263.02) < 0.01      # BASELINE.md section 3
    assert abs(f3["conv"] + f3["wgrad"] - f3["step"]) < 1
    # 69 dense blocks carry 92 % of the generator forward (SURVEY.md 8a row a1: 16.93 of 18.37 GMAC)
    assert abs(bench.N_RDB * bench.F_RDB / 1e9 - 2 * 16.93) < 0.01
    assert abs(256 * f3["infer_per_chunk"] / 1e12 - 9.405) < 0.001                                # per 2048^2 tile
    c12, lr12 = bench.train_config(12), bench.synthetic_batch(2, 0, bands=12)[0]
    assert c12["num_in_ch_g"] == 96 and c12["num_in_ch_d"] == 99 and lr12.shape == (2, 96, 32, 32)
    opt = bench.model_opt(12, True, False)
    assert opt["network_g"]["num_in_ch"] == 96 and opt["network_d"]["num_in_ch"] == 99 and opt["model_type"] == "SSRESRGANModel"
    # the roofline block from a measured dict (numbers of profiles/r02c_logs/bench_default_final.json): dominant kernel = resident dense blocks
    m = dict(B=32, ms_cls=[5.9, 1.7, 2.84, 2.58, 2.2], cnt_cls=[130, 26, 6, 6, 69], side_lane=True,
             graph_us={"forward": {"launches": 6, "us_per_launch": 446.3}, "input_gradient": {"launches": 6, "us_per_launch": 403.0}})
    main, others = bench.train_rooflines(m, 3, 1452.2, "measured")
    assert main["bound"] == "tensor" and main["unit"] == "TFLOP/s" and abs(main["frac"] - main["achieved"] / 1452.2) < 1e-9
    assert 0.26 < main["frac"] < 0.29 and main["launches_per_step"] == 12 and "side lane" in main["timing"]
    assert abs(main["forward"]["in_graph"]["us_per_block"] - 446.3 * 6 / 69) < 1e-6 and 0.30 < main["input_gradient"]["in_graph"]["frac"] < 0.32
    assert main["traffic"] and main["traffic"] > 1e8        # per 12-block launch, from profiles/ncu_traffic.json (ncu --set full)
    assert set(others) == {"conv_tc_kernel", "wgrad9_tc_batched_kernel", "wgrad_tc_kernels", "all_conv_fwd_dgrad"}
    assert "side lane" not in bench.train_rooflines(dict(m, side_lane=False, graph_us={}), 3, 1452.2, "measured")[0]["timing"]


def format_s2naip_input():
    import numpy as np
    rng = np.random.RandomState(0)
    s2 = rng.randint(1, 255, size=(10 * 32, 32, 3)).astype(np.uint8)
    s2[3 * 32 + 5, 7] = 0                       # frame 3 has a pure-black pixel -> "bad"
    return s2


def test_infer_format_matches_reference_semantics():
    import random
    import numpy as np
    from satlas_super_resolution_b200.infer import format_s2naip_data
    s2 = format_s2naip_input()
    t, first = format_s2naip_data(s2, 8, rng=random.Random(1))
    assert t.shape == (1, 24, 32, 32) and t.dtype == torch.float32 and float(t.max()) <= 1
    assert np.array_equal(first, s2[:32])
    # bad frames are only used when there are not enough good ones
    frames = {tuple(s2[i * 32:(i + 1) * 32].transpose(2, 0, 1).flatten()[:8]) for i in range(10) if i != 3}
    for k in range(8):
        assert tuple((t[0, 3 * k:3 * k + 3] * 255).round().byte().numpy().flatten()[:8]) in frames
    # what the reference's format_s2naip_data returned for this input after random.seed(5) (oracle/make_golden_ref.py)
    gold = torch.load(os.path.join(ROOT, "tests", "golden", "format_s2naip_data.pt"))
    got, got_first = format_s2naip_data(s2, gold["n_s2_images"], rng=random.Random(gold["random_seed"]))
    assert torch.equal(gold["s2_tensor_u8"].float() / 255, got) and np.array_equal(gold["s2_image"].numpy(), got_first)


GLOO_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from collections import OrderedDict
from satlas_super_resolution_b200.ops import FlatBuffer, allreduce_sum_, broadcast_from_rank0_, rank_slice
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
# replicas initialised from rank-dependent seeds (ssr/utils/options.py:81: manual_seed + rank) end up with rank 0's state: what
# DistributedDataParallel does to parameters and buffers at construction (ESRGANTrainer.sync_replicas)
torch.manual_seed(100 + rank)
params, u = FlatBuffer(OrderedDict(w=(4, 3), b=(5,)), "cpu"), torch.randn(7)
params.flat.normal_()
broadcast_from_rank0_([params.flat, u], dist.group.WORLD)
torch.manual_seed(100)
want_u = torch.randn(7)
want = torch.empty_like(params.flat).normal_()
assert torch.equal(params.flat, want) and torch.equal(u, want_u), "replica state differs from rank 0 after the broadcast"
shapes = OrderedDict(w=(4, 3), b=(5,))
g = FlatBuffer(shapes, "cpu")
# per-rank "gradient" = mean over this rank's shard of per-sample gradients
torch.manual_seed(0)
per_sample = torch.randn(8, g.numel)
mine = per_sample[list(rank_slice(8, rank, world))].mean(0)
g.flat.copy_(mine)
allreduce_sum_(g.flat, dist.group.WORLD)
avg = g.flat / world                     # the 1/world the fused Adam kernel applies as grad_scale
assert torch.allclose(avg, per_sample.mean(0), atol=1e-6), "sharded average != big-batch average"
# loss scalars: reduce to rank 0 and divide (trainer.get_current_log)
t = torch.tensor([float(rank + 1), 2.0])
dist.reduce(t, dst=0)
if rank == 0:
    assert torch.allclose(t / world, torch.tensor([1.5, 2.0]))
# the step's exchange schedule (ESRGANTrainer._run_step): G gradients are exchanged asynchronously after phase 1 and summed before
# phase 3 (Adam(G)), D gradients after phase 2 and before phase 4 (Adam(D)); without a generator step only D is exchanged
from satlas_super_resolution_b200.trainer import ESRGANTrainer
class Stub:
    pass
st = Stub()
st.world, st.pg = world, dist.group.WORLD
st.ggrad, st.dgrad = FlatBuffer(shapes, "cpu"), FlatBuffer(OrderedDict(d=(6,)), "cpu")
st._exchange_async = ESRGANTrainer._exchange_async.__get__(st)
for do_g in (True, False):
    log = []
    def run_phase(ph):
        log.append(ph)
        if ph == 1:
            st.ggrad.flat.fill_(float(rank + 1))
        elif ph == 2:
            st.dgrad.flat.fill_(10.0 * (rank + 1))
        elif ph == 3:
            want = 3.0 if do_g else float(rank + 1)          # 1 + 2 summed over the two ranks, or untouched
            assert torch.all(st.ggrad.flat == want), (do_g, st.ggrad.flat)
        elif ph == 4:
            assert torch.all(st.dgrad.flat == 30.0), st.dgrad.flat
    ESRGANTrainer._run_step(st, run_phase, do_g)
    assert log == [1, 2, 3, 4]
dist.barrier()
dist.destroy_process_group()
print("gloo-ok", rank)
'''


def test_gradient_exchange_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"gloo-ok {r}" in o, o


def test_missing_vgg19_checkpoint_is_an_error_unless_random_weights_are_requested(tmp_path, monkeypatch):
    """basicsr loads the ImageNet VGG19 (downloading when absent); silently training against random features would be a
    meaningless perceptual term (ADVICE round 1): missing file -> FileNotFoundError, explicit vgg_seed -> seeded weights + warning"""
    from satlas_super_resolution_b200 import weights
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("TORCH_HOME", str(tmp_path / "no_hub"))
    monkeypatch.delenv("SSR_VGG19_PATH", raising=False)
    monkeypatch.delenv("SSR_VGG_RANDOM_SEED", raising=False)
    with pytest.raises(FileNotFoundError):
        weights.resolve_vgg19_state()
    with pytest.warns(RuntimeWarning):
        sd = weights.resolve_vgg19_state(vgg_seed=3)
    assert torch.equal(sd["conv3_2.weight"], weights.vgg19_state(seed=3)["conv3_2.weight"])
    # a checkpoint in torchvision's layout at $SSR_VGG19_PATH is picked up
    raw = {}
    for (name, cin, cout), idx in zip(weights.VGG19_CONVS, weights.VGG19_TORCHVISION_INDEX):
        raw[f"features.{idx}.weight"] = torch.full((cout, cin, 3, 3), float(idx))
        raw[f"features.{idx}.bias"] = torch.zeros(cout)
    torch.save(raw, tmp_path / "vgg.pth")
    monkeypatch.setenv("SSR_VGG19_PATH", str(tmp_path / "vgg.pth"))
    sd = weights.resolve_vgg19_state()
    assert sd["conv5_4.weight"][0, 0, 0, 0].item() == 34.0


def test_load_tile_dir_matches_the_reference_frame_choice(tmp_path):
    """infer.load_tile_dir (threaded PNG decode of one {tile}/{i}_{j}.png directory): the chunk stack equals what the reference's
    format_s2naip_data (ssr/utils/infer_utils.py:6-39, restated in infer.format_s2naip_data) yields chunk by chunk under the same
    seeded `random`, and the stitched first frames equal stitch(..., sentinel2=True) (infer_utils.py:41-60)."""
    import random
    from concurrent.futures import ThreadPoolExecutor
    import cv2
    import numpy as np
    from satlas_super_resolution_b200.infer import format_s2naip_data, load_tile_dir
    rs = np.random.RandomState(0)
    grid, T, n = 3, 6, 4
    d = tmp_path / "tile_a"
    d.mkdir()
    ims = {}
    for i in range(grid):
        for j in range(grid):
            im = rs.randint(1, 256, (T * 32, 32, 3)).astype(np.uint8)
            if (i + j) % 2:                       # some frames with black pixels: used only when clean ones run out
                im[0:32][5, 7] = 0
                im[64:96][0, 0] = 0
                im[96:128][1, 1] = 0
            ims[(i, j)] = im
            cv2.imwrite(str(d / f"{i}_{j}.png"), cv2.cvtColor(im, cv2.COLOR_RGB2BGR))
    with ThreadPoolExecutor(4) as pool:
        stack, s2 = load_tile_dir(str(d), n, grid_size=grid, pool=pool, rng=random.Random(7))
    rng = random.Random(7)
    for k in range(grid * grid):
        i, j = divmod(k, grid)
        want, first = format_s2naip_data(ims[(i, j)], n, rng=rng)
        assert torch.equal(stack[k].float() / 255, want[0])
        assert np.array_equal(s2[i * 32:(i + 1) * 32, j * 32:(j + 1) * 32], first)
    assert stack.shape == (grid * grid, n * 3, 32, 32) and stack.dtype == torch.uint8


def test_plan_lanes_order_forks_and_joins():
    """Plan (ops.py): calls recorded inside plan.side() go to the side lane; fork / join are replayed where they were recorded and run()
    joins at its end (a CUDA-graph capture must not end with an unjoined stream)."""
    from satlas_super_resolution_b200.ops import Plan
    log = []

    class Lane:
        handle = "side"

        def fork(self, s):
            log.append(("fork", s))

        def join(self, s):
            log.append(("join", s))

    def k(name):
        def fn(*args):
            log.append((name, args[-1]))
            return 0
        return fn

    plan = Plan()
    plan.add(k("chain0"), 1)
    plan.fork()
    with plan.side():
        plan.add(k("wgrad0"), 2)
    plan.add(k("chain1"), 3)
    plan.join()
    plan.fork()
    with plan.side():
        plan.add(k("wgrad1"), 4)
    plan.add(k("tail"), 5)
    assert plan.has_side and len(plan) == 5 and [c[0].__name__ for c in plan.main_calls()] == ["fn"] * 3
    plan.run("main", lane=Lane())
    assert log == [("chain0", "main"), ("fork", "main"), ("wgrad0", "side"), ("chain1", "main"), ("join", "main"), ("fork", "main"),
                   ("wgrad1", "side"), ("tail", "main"), ("join", "main")]
    # a plan without side calls never touches a lane
    log.clear()
    p2 = Plan()
    p2.add(k("a"), 0)
    p2.run("main", lane=None)
    assert log == [("a", "main")] and not p2.has_side
    # a failing call raises through L.check
    p3 = Plan()
    with p3.side():
        p3.add(lambda *a: 1, 0)
    with pytest.raises(Exception):
        p3.run("main", lane=Lane())


def test_side_lane_switch_parsing(monkeypatch):
    """ops.overlap_enabled: option value first, then $SSR_OVERLAP, default on; 'fwd' / 'bwd' select one part"""
    from satlas_super_resolution_b200.ops import overlap_enabled as on
    monkeypatch.delenv("SSR_OVERLAP", raising=False)
    assert on() and on("fwd") and on("bwd")
    assert not on("fwd", False) and on("bwd", True) and on("fwd", "fwd") and not on("bwd", "fwd") and on("bwd", "fwd,bwd")
    assert not on(None, "0") and not on("bwd", "off") and on(None, "bwd")
    monkeypatch.setenv("SSR_OVERLAP", "0")
    assert not on() and not on("fwd") and on("fwd", True)          # an explicit option overrides the environment
    monkeypatch.setenv("SSR_OVERLAP", "bwd")
    assert on("bwd") and not on("fwd")
