#!/usr/bin/env python
"""bench.py -- occupancy Mpoints/s (+ recon frames/s @256^3) of the fused hot path on N B200s of one node.

    python bench.py --gpus 1 --steps K --warmup W
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        (the reference's CPU path: the oracle port, host cores)
    python bench.py ... --dump-outputs DIR      (also writes the last timed step's occupancy volume, see dump_volume)

A "step" = one pass of the hot path over one synthetic frame: upload-free channel-last repack of the [1,256,128,128]
feature map + the fused sample+MLP kernel over the dense 257^3 node grid ("256^3", RTL/main.py:187), z-slab
sharded over the ranks, + ONE all-gather of the occupancy volume (N>1).  `value` = whole-job Mpoints/s with inputs
resident in HBM; `e2e` = the same through the C-ABI host-buffer entry point (feature map H2D + volume D2H inside the
timed region; at N > 1 the all-gather too).  `recon` reports BASELINE configs[1..3] (coarse-to-fine recon frames/s, with the
netC colour pass, and the image stream with the PyTorch encoder as CUDA-graph captured frame steps), `configs4_dense513`
BASELINE configs[4].  At N > 1 the line also asserts that the gathered volume equals the single-GPU volume bit for bit.
Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

R_GRID = 257
FLOP_PER_POINT = 2363906          # 2*(257*1024+1281*512+769*256+513*128+385*1)  (BASELINE.md §4)
# DRAM bytes of one query_tc3_kernel launch over the dense 257^3 grid, from an `ncu --set full` capture (not re-measured by a
# bench run: profiling and timing never share a run).  Updated by hand from profiles/ when the kernel changes.
TRAFFIC_NCU = {"bytes": 82.69e6, "source": "profiles/r02_final_ncu_tc_summary.txt: 44.79 MB read + 37.90 MB written (ncu --set full pass of tools/gpu_r02_final.sh)"}
B_MIN, B_MAX = (-1.0, -1.0, -1.0), (1.0, 1.0, 1.0)
DUMP_NODES = 1 << 22              # --dump-outputs: a volume with more nodes is sampled (16 MB of values + 32 MB of node ids)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=os.environ.get("MONOPORT_B200_MODE", "auto"), choices=["auto", "tc", "fp32"])
    ap.add_argument("--res", type=int, default=R_GRID)
    ap.add_argument("--exchange", default=os.environ.get("MONOPORT_B200_EXCHANGE", "auto"), choices=["auto", "nccl", "fused"],
                    help="N>1, how the ranks' ranges become the volume on every rank: 'nccl' = one in-place all-gather, 'fused' = "
                         "peer-memory stores from the kernel epilogue + a barrier; 'auto' = fused from 4 GPUs on (measured: 2 GPUs "
                         "1101 vs 1086 Mpoints/s in favour of NCCL, 8 GPUs 4647 vs 4733 in favour of the fused exchange)")
    ap.add_argument("--fused-gather", action="store_true", help="same as --exchange fused")
    ap.add_argument("--no-recon", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the occupancy volume of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(source="measured", tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm=d["hbm_gbs"])
    return dict(source="fallback", tf_burst=1590.0, tf_sustained=1400.0, hbm=6650.0)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def synthetic(seed_w=3, seed_f=4, n_feat=1):
    """Seeded random-init netG head + feature maps of the encoder's shape; the 'person' wiring keeps the cost per
    point unchanged (oracle/spec.py:heightfield_person is test infra -- the same construction is inlined here so
    that the product bench does not import the oracle)."""
    import math
    import torch
    chans = [257, 1024, 512, 256, 128, 1]
    g = torch.Generator().manual_seed(seed_w)
    Ws, bs = [], []
    for l in range(5):
        cin = chans[l] + (chans[0] if l else 0)
        k = 1.0 / math.sqrt(cin)
        Ws.append((torch.rand(chans[l + 1], cin, generator=g) * 2 - 1) * k)
        bs.append((torch.rand(chans[l + 1], generator=g) * 2 - 1) * k)
    feats = []
    H = W = 128
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, H), torch.linspace(-1, 1, W), indexing="ij")
    for i in range(n_feat):
        gf = torch.Generator().manual_seed(seed_f + i)
        f = torch.randn(1, 256, H, W, generator=gf) * 0.5
        body = 1 - ((xx / 0.28) ** 2 + ((yy - 0.05) / 0.62) ** 2)
        head = 1 - ((xx / 0.16) ** 2 + ((yy + 0.68) / 0.17) ** 2)
        arm = 1 - (((xx.abs() - 0.40) / 0.10) ** 2 + ((yy + 0.05 - 0.02 * i) / 0.40) ** 2)
        f[0, 0] = torch.maximum(torch.maximum(body, head), arm).clamp(min=-1.0) * 0.35
        feats.append(f.contiguous())
    C = 256
    Ws[3][0].zero_(); Ws[3][1].zero_()
    Ws[3][0, 256 + C] = 1.0; Ws[3][1, 256 + C] = -1.0
    bs[3][0] = 0.0; bs[3][1] = 0.0
    Ws[4].zero_(); bs[4].zero_()
    Ws[4][0, 128 + 0] = 40.0
    Ws[4][0, 0] = -40.0 / 0.99; Ws[4][0, 1] = -40.0 / 0.99
    return chans, Ws, bs, feats


def scene_calib():
    """pifu_calib of the demo camera at yaw 20 deg, pitch 33 deg (RTL/scene.py:108-135, RTL/recon.py:4-25)."""
    import math
    import numpy as np
    from monoport_b200.recon import pifu_calib

    def rot(rx, ry):
        cx, sx, cy, sy = math.cos(rx), math.sin(rx), math.cos(ry), math.sin(ry)
        Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
        Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        return Ry @ Rx
    E = np.eye(4)
    E[:3, :3] = rot(math.radians(20), 0) @ rot(0, math.radians(33))
    E[:3, 3] = [0, 0, -2.0]
    K = np.diag([1.0, 1.0, -0.2, 1.0]); K[2, 3] = -1.0
    return pifu_calib(E, K, device="cpu")


def dump_volume(dirname, vol):
    """--dump-outputs: the volume as `volume.npy` (float32, z-major [R,R,R]) when it has at most DUMP_NODES nodes, else a fixed
    seeded sample of DUMP_NODES nodes as `volume_sample.npy` (float32) with their linear z-major node ids in
    `volume_sample_node.npy` (float64), so that two builds can be compared value for value."""
    import numpy as np
    import torch
    if vol.numel() <= DUMP_NODES:
        arrays = {"volume": vol}
    else:
        node = torch.randint(0, vol.numel(), (DUMP_NODES,), generator=torch.Generator().manual_seed(29))
        arrays = {"volume_sample": vol.reshape(-1)[node.to(vol.device)], "volume_sample_node": node.double()}
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a.cpu().numpy())


# ------------------------------------------------------------------------------------------------------------
def best_threads(fn):
    """The torch-CPU port does not scale to every hardware thread of a big host: time a small sample at a few thread
    counts and keep the fastest (reported as `cores`)."""
    import torch
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores // 2, cores) if 1 <= c <= cores})
    best, best_t = cores, None
    for c in cands:
        torch.set_num_threads(c)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def run_reference(args):
    """The reference's own CPU implementation of the path = the oracle port (the Python reference cannot travel
    to the GPU box), all host threads, on a bounded sample of the same workload per step."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import spec
    chans, Ws, bs, feats = synthetic()
    cal = scene_calib()
    S = 48                                                  # 48^3 = 110 592 node centres of the same [-1,1]^3 grid
    coords = spec._grid_coords(S, 1)
    pts = spec.level_points(coords, S, B_MIN, B_MAX).t().contiguous()
    cores = best_threads(lambda: spec.query_ref(feats[0], pts[:, :16384], cal, Ws, bs, spec.LAST_SIGMOID))
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        occ = spec.query_ref(feats[0], pts, cal, Ws, bs, spec.LAST_SIGMOID)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_volume(args.dump_outputs, occ.reshape(S, S, S))
    total = sum(times)
    mpts = S ** 3 * len(times) / total / 1e6
    line = {
        "impl": "reference", "metric": "occupancy_mpoints_per_s", "value": mpts, "unit": "Mpoints/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "netG query() over dense grid node centres, [1,256,128,128] features, scene calib "
                               "yaw20/pitch33; bounded sample 48^3 = 110592 points per step of the 257^3 job"},
        "cpu_baseline": {"value": mpts, "unit": "Mpoints/s", "cores": cores, "kind": "port",
                         "sample": "48^3 = 110592 points per step, torch CPU fp32, %d threads" % cores},
        "e2e": {"value": mpts, "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def _person_hook(height):
    """Stream workload: the encoder's last-stage map with channel 0 replaced by a synthetic body height map, so that the
    frame (points evaluated, vertices) is the same in every run -- the random-init encoder alone gives a noise surface."""
    def hook(f):
        f = f.clone()
        f[:, 0] = height
        return f
    return hook


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from monoport_b200 import _lib
    from monoport_b200.modeling import PIFuNetG
    from monoport_b200.shard import ShardedVolume, PeerVolumes, query_grid_fused, range_bounds

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 through torch.distributed.run (see docstring)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)

    R = args.res
    chans, Ws, bs, feats_cpu = synthetic(n_feat=4)
    torch.manual_seed(0)                       # the encoder's random init (stream workload) is the same in every run
    net = PIFuNetG()
    net.surface_classifier.load_state_dict(
        {**{"filters.%d.weight" % l: W[:, :, None] for l, W in enumerate(Ws)},
         **{"filters.%d.bias" % l: b for l, b in enumerate(bs)}})
    net.surface_classifier.to(dev)
    net.eval()
    net.precision = args.mode
    mode_used = "tc" if (args.mode in ("auto", "tc") and net.surface_classifier.tc_supported()) else "fp32"
    if args.mode == "tc" and mode_used != "tc":
        raise SystemExit("tcgen05 kernel unavailable")
    cal_cpu = scene_calib()
    cal = cal_cpu.to(dev)
    feats = [f.to(dev) for f in feats_cpu]
    n_pts_total = R ** 3
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2
    # balanced ranges of the z-major node order (z slabs whose boundaries need not fall on planes), ONE in-place all-gather
    sv = ShardedVolume(R, rank, world, dev)
    lin0, my_pts = sv.bounds[rank]

    exchange = "fused" if args.fused_gather else args.exchange
    if exchange == "auto":
        exchange = "fused" if world >= 4 else "nccl"
    fused = bool(exchange == "fused" and world > 1)
    peers = PeerVolumes(R, rank, world, dev) if fused else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(i, fh=None):
        f = feats[i % len(feats)]
        if fused:
            return query_grid_fused(net, f, cal_cpu, R, B_MIN, B_MAX, peers, fh=fh)
        sv.query(net, f, cal_cpu, B_MIN, B_MAX, fh=fh)
        return None

    for i in range(args.warmup):
        step(i)
        if not fused:
            sv.gather()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    vol = None
    for i in range(args.steps):
        flush.fill_(float(i))                      # L2 flush between timed iterations (not timed)
        f = feats[i % len(feats)]
        ev[i][0].record()
        fh = net.feature_handle(f)                 # channel-last repack kernel (part of the step)
        kev[i][0].record()
        vol = step(i, fh)                          # fused: kernel with peer stores + barrier
        kev[i][1].record()
        if not fused:
            vol = sv.gather()                      # N > 1: one in-place all-gather inside the persistent buffer
        ev[i][1].record()
    barrier()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_volume(args.dump_outputs, vol)
    t_ms = sum(a.elapsed_time(b) for a, b in ev)
    k_ms = sum(a.elapsed_time(b) for a, b in kev)
    tt = torch.tensor([t_ms, k_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_ms, k_ms = tt.tolist()
    value = n_pts_total * args.steps / (t_ms * 1e-3) / 1e6

    # ---- what was timed is right: the volume every rank holds == the volume ONE GPU computes, bit for bit; and the
    #      tensor-core values agree with the exact fp32 kernel on a sample of the same grid -------------------------
    f_last = feats[(args.steps - 1) % len(feats)]
    single = net.query_grid(f_last, cal_cpu, R, B_MIN, B_MAX) if world > 1 else vol
    same = torch.tensor([int(torch.equal(vol, single))], device=dev)
    if world > 1:
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
    volume_ok = bool(same.item())
    checksum = float(vol.double().sum().item())
    g = torch.Generator().manual_seed(17)
    lin = torch.randint(0, R ** 3, (16384,), generator=g)
    parity = None
    if mode_used == "tc":
        R_f = float(R)
        xyz = torch.stack([(lin % R).float(), ((lin // R) % R).float(), (lin // (R * R)).float()], 0)
        pts = (((xyz / R_f) + 1.0 / (2.0 * R_f)) * 2.0 - 1.0)[None].to(dev)          # node centres, [1,3,N]
        net.precision = "fp32"
        exact = net.query([[f_last]], pts, calibs=cal_cpu)[0]
        net.precision = args.mode
        parity = float((vol.reshape(-1)[lin.to(dev)] - exact[0, 0]).abs().max().item())
    del single

    # ---- e2e through the C-ABI with HOST buffers (pinned): feature map H2D, this rank's range of the volume D2H, and --
    #      at N > 1 -- the all-gather in between (the job's result is the assembled volume) ---------------------------
    lib = _lib.load()
    feat_pinned = [f.pin_memory() for f in feats_cpu]
    out_host = torch.empty(max(my_pts, 1), dtype=torch.float32).pin_memory()
    fh = net.feature_handle(feats[0])
    cal12 = _lib.calib12(cal_cpu)
    st = _lib.stream_ptr(dev)
    mode_code = _lib.MODE_TC if mode_used == "tc" else _lib.MODE_FP32

    def e2e_step(i):
        f = feat_pinned[i % len(feat_pinned)]
        if world == 1:
            _lib.check(lib.mp_query_grid_host(net.surface_classifier.handle(), fh.ptr, ctypes.c_void_p(f.data_ptr()), R, 0, R,
                                              _lib.f3(B_MIN), _lib.f3(B_MAX), cal12, 0, ctypes.c_float(net.normalizer.scale),
                                              ctypes.c_void_p(out_host.data_ptr()), mode_code, st))
            return
        _lib.check(lib.mp_feat_upload(fh.ptr, ctypes.c_void_p(f.data_ptr()), 0, st))                      # H2D + repack
        _lib.check(lib.mp_query_grid_range(net.surface_classifier.handle(), fh.ptr, R, lin0, my_pts, _lib.f3(B_MIN), _lib.f3(B_MAX),
                                           cal12, 0, ctypes.c_float(net.normalizer.scale), ctypes.c_void_p(sv.segment.data_ptr()),
                                           mode_code, st))
        sv.gather()
        out_host[:my_pts].copy_(sv.segment[:my_pts], non_blocking=True)                                     # D2H
        torch.cuda.current_stream().synchronize()
    e2e_steps = max(3, min(args.steps, 10))
    e2e_step(0)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = n_pts_total * e2e_steps / te.item() / 1e6
    fh.key = None

    # ---- configs[1..3]: coarse-to-fine recon frames/s -------------------------------------------------------------
    recon = None
    if not args.no_recon and R == R_GRID:
        recon = bench_recon(args, net, feats, cal, cal_cpu, dev, rank, world, barrier)
    # ---- configs[4]: dense 513^3 ("512^3") through the same sharded step, a few steps ------------------------------
    c4 = None
    if not args.no_recon and R == R_GRID:
        R5 = 513
        sv5 = ShardedVolume(R5, rank, world, dev)
        for i in range(1):
            sv5.query(net, feats[0], cal_cpu, B_MIN, B_MAX); sv5.gather()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n5 = 3
        e0.record()
        for i in range(n5):
            sv5.query(net, feats[i % 4], cal_cpu, B_MIN, B_MAX); v5 = sv5.gather()
        e1.record()
        barrier()
        t5 = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t5, op=dist.ReduceOp.MAX)
        c4 = {"workload": "configs[4]: netG dense 513^3 (135 005 697 points), range-sharded over %d GPU(s) + 1 all-gather (540 MB volume)" % world,
              "ms_per_volume": t5.item() / n5, "mpoints_per_s": R5 ** 3 * n5 / (t5.item() * 1e-3) / 1e6,
              "occupied_fraction": float((v5 > 0.5).float().mean().item())}
        del sv5, v5

    # ---- CPU baseline (reported, not the target): the oracle port on a bounded sample, rank 0, N=1 only ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import spec
        S = 64                                                     # BASELINE configs[0]: dense 64^3 on CPU
        pts = spec.level_points(spec._grid_coords(S, 1), S, B_MIN, B_MAX).t().contiguous()
        cores = best_threads(lambda: spec.query_ref(feats_cpu[0], pts[:, :16384], cal_cpu, Ws, bs, spec.LAST_SIGMOID))
        t0 = time.perf_counter()
        reps = 0
        ref = None
        while time.perf_counter() - t0 < 10.0 or reps < 1:
            ref = spec.query_ref(feats_cpu[0], pts, cal_cpu, Ws, bs, spec.LAST_SIGMOID)
            reps += 1
        dt = time.perf_counter() - t0
        ours64 = net.query([[feats[0]]], pts[None].to(dev), calibs=cal_cpu)[0][0].cpu()
        cpu = {"value": S ** 3 * reps / dt / 1e6, "unit": "Mpoints/s", "cores": cores, "kind": "port",
               "sample": "dense 64^3 = 262144 points x %d reps (%.1f s), torch CPU fp32 oracle port of MonoPortNet.query" % (reps, dt),
               "parity_max_abs_vs_oracle": float((ours64 - ref).abs().max().item())}

    if rank == 0:
        pk = peaks()
        # nchw_to_nhwc repack + per-texel layer-0 GEMM (g0_tc_kernel) + fused query kernel + the range guard's (empty) exact-kernel launch
        launches_per_step = 4 if mode_used == "tc" else 2
        k_avg_s = k_ms * 1e-3 / args.steps
        achieved_tf = FLOP_PER_POINT * my_pts / k_avg_s / 1e12
        peak_tf = pk["tf_sustained"]
        line = {
            "metric": "occupancy_mpoints_per_s", "value": value, "unit": "Mpoints/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f16" if mode_used == "tc" else "f32", "data": "synthetic",
            "config": {"workload": "netG dense %d^3 grid query (%d points/step), [1,256,128,128] features, scene calib "
                                   "yaw20/pitch33, balanced z-major ranges over %d GPU(s) + %s" % (R, n_pts_total, world, "peer-memory stores from the kernel epilogue + 1 barrier" if fused else "1 in-place all-gather"),
                       "kernel_mode": mode_used, "l2_flush_between_steps": True, "grid": R,
                       "accumulate": "fp32", "last_layer": "fp32"},
            "volume_matches_single_gpu": volume_ok, "volume_checksum": checksum,
            "parity_max_abs": parity, "parity_note": "tensor-core volume vs the exact fp32 kernel on 16384 random nodes of this grid (bar 1e-4); cpu_baseline.parity_max_abs_vs_oracle: vs the oracle on the 64^3 sample",
            "e2e": {"value": e2e_value, "unit": "Mpoints/s", "h2d_bytes_per_step": 256 * 128 * 128 * 4 + 48,
                    "d2h_bytes_per_step": my_pts * 4, "steps": e2e_steps,
                    "api": "mp_query_grid_host (pinned host feature map in, host occupancy volume out)" if world == 1 else
                           "mp_feat_upload(host) + mp_query_grid_range + all-gather + D2H of this rank's range"},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak_tf,
                         "traffic": (TRAFFIC_NCU["bytes"] if (mode_used == "tc" and world == 1 and R == R_GRID) else None),
                         "traffic_unit": "bytes/launch, dram__bytes_read.sum + dram__bytes_write.sum of query_tc3_kernel (%s)" % TRAFFIC_NCU["source"],
                         "kernel": ("query_tc3_kernel (+ g0_tc_kernel, the per-frame per-texel layer-0 GEMM, 25 us)" if mode_used == "tc"
                                    else "query_fp32_kernel"),
                         "kernel_ms": 1e3 * k_avg_s, "peak_source": pk["source"] + " bf16 sustained (cuBLAS loop)",
                         "frac_of_burst": achieved_tf / pk["tf_burst"],
                         "algorithmic_flop_per_point": FLOP_PER_POINT},
            "clocks": clocks,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if recon:
            line["recon"] = recon
        if c4:
            line["configs4_dense513"] = c4
        print(json.dumps(line))
    if peers is not None:
        barrier()
        peers.close()
    if world > 1:
        dist.destroy_process_group()


def bench_recon(args, net, feats, cal, cal_cpu, dev, rank, world, barrier):
    """configs[1] (coarse-to-fine recon, one image), configs[2] (+ netC colour), configs[3] (image stream) -- per rank at N = 1,
    and at N > 1: frame-parallel replicas (every rank reconstructs its own frames) and the list-sharded engine."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from monoport_b200.engine import Seg3dLossless, make_query_func
    from monoport_b200.recon import forward_vertices, marching_cubes, colorization
    from monoport_b200.pipeline import FrameGraph, FrameGraphRing
    b = np.array([B_MIN], dtype=np.float32)
    res = [17, 33, 65, 129, 257]
    eng = Seg3dLossless(make_query_func(net), b, -b, res, balance_value=0.5, faster=True).to(dev)
    out = {"workload": "netG 256^3 Seg3dLossless(faster=True) on a body-like height field, per frame"}

    def timed(fn, n):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(n):
            fn(i)
        torch.cuda.synchronize()
        return n / (time.perf_counter() - t0)

    nfr = 20
    if world == 1:
        for i in range(3):                                  # warm-up: engine, surface kernel, marching cubes
            sdf = eng(im_feat_list=[[feats[i % 4]]], calib_tensor=cal_cpu)
            X, Y, Z, nrm = forward_vertices(sdf, "front")
            v, fcs = marching_cubes(sdf[0, 0])
        state = {}

        def fv(i):
            state["sdf"] = eng(im_feat_list=[[feats[i % 4]]], calib_tensor=cal_cpu)
            state["fv"] = forward_vertices(state["sdf"], "front")

        def mc(i):
            sdf_ = eng(im_feat_list=[[feats[i % 4]]], calib_tensor=cal_cpu)
            state["mesh"] = marching_cubes(sdf_[0, 0])
        out["frames_per_s_with_forward_vertices"] = timed(fv, nfr)
        out["frames_per_s_with_marching_cubes"] = timed(mc, nfr)
        recon_stats = list(eng.last_stats)
        X, Y, Z, nrm = state["fv"]
        v, fcs = state["mesh"]
        # the same frame as ONE CUDA-graph launch (pipeline.FrameGraph), one and two lanes
        for lanes in (1, 2, 4):
            ring = FrameGraphRing(lambda: FrameGraph(net, eng, cal_cpu, "front", with_encoder=False), n_lanes=lanes)
            list(ring.run(feats[i % 4] for i in range(4)))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n_g = 60
            for r_ in ring.run(feats[i % 4] for i in range(n_g)):
                pass
            torch.cuda.synchronize()
            out["frames_per_s_frame_graph_%d_lane%s" % (lanes, "s" if lanes > 1 else "")] = n_g / (time.perf_counter() - t0)
            ring.close()
        # configs[2]: geometry + colour -- netC queried at the visible vertices, fused direct rendering (tensor-core colour program)
        from monoport_b200.modeling import PIFuNetC
        netC = PIFuNetC()
        netC.surface_classifier.to(dev)
        netC.eval()
        gC = torch.Generator().manual_seed(11)
        featC = [[(torch.randn(1, 512, 128, 128, generator=gC) * 0.5).to(dev)]]
        colorization(netC, featC, X, Y, Z, cal)

        def col(i):
            sdf_ = eng(im_feat_list=[[feats[i % 4]]], calib_tensor=cal_cpu)
            X_, Y_, Z_, _n = forward_vertices(sdf_, "front")
            state["img"] = colorization(netC, featC, X_, Y_, Z_, cal)
        out["frames_per_s_geometry_plus_netC_colour"] = timed(col, nfr)
        out.update({"points_evaluated_per_frame": int(sum(recon_stats)), "per_level": recon_stats,
                    "visible_vertices": int(X.numel()), "mesh_vertices": int(v.shape[0]), "mesh_faces": int(fcs.shape[0])})
    # configs[3]: image stream -- synthetic 512x512 frames -> HG encoder (PyTorch fp32) -> recon -> visible surface, every frame
    # one CUDA-graph launch, two lanes in flight per GPU; at N > 1 the ranks work on different frames (frame-parallel replicas)
    net.image_filter.to(dev)
    gI = torch.Generator().manual_seed(5 + rank)
    frames = [(torch.rand(1, 3, 512, 512, generator=gI) * 2 - 1).to(dev) for _ in range(4)]
    hook = _person_hook(feats[0][:, 0].clone())
    stream = {}
    for lanes in (1, 2, 3):
        ring = FrameGraphRing(lambda: FrameGraph(net, eng, cal_cpu, "front", with_encoder=True, feature_hook=hook), n_lanes=lanes)
        list(ring.run(frames[i % 4] for i in range(4)))
        barrier()
        t0 = time.perf_counter()
        nst = 40
        for r_ in ring.run(frames[i % 4] for i in range(nst)):
            pass
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        stream["%d_lane%s" % (lanes, "s" if lanes > 1 else "")] = world * nst / dt.item()
        pts_frame = int(sum(ring.lanes[0].last_stats))
        ring.close()
    out["configs3_stream_frames_per_s"] = dict(stream, note="512x512 frame -> HGFilter (PyTorch fp32, seeded random init; channel 0 of its map carries the synthetic "
                                               "body height field, %d points evaluated per frame) -> recon -> forward_vertices; one CUDA-graph launch per frame "
                                               "(pipeline.FrameGraph); %d GPU(s) = frame-parallel replicas" % (pts_frame, world))
    if world > 1:
        # the list-sharded engine: ONE frame at a time over all GPUs (MLP evaluations split, volume passes replicated)
        sh = Seg3dLossless(make_query_func(net), b, -b, res, balance_value=0.5, faster=True).to(dev).shard(rank, world)
        for i in range(3):
            sdf = sh(im_feat_list=[[feats[i % 4]]], calib_tensor=cal_cpu)
        barrier()
        t0 = time.perf_counter()
        for i in range(nfr):
            sdf = sh(im_feat_list=[[feats[i % 4]]], calib_tensor=cal_cpu)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        single = eng(im_feat_list=[[feats[(nfr - 1) % 4]]], calib_tensor=cal_cpu)
        okv = torch.tensor([int(torch.equal(sdf, single))], device=dev)
        dist.all_reduce(okv, op=dist.ReduceOp.MIN)
        out["list_sharded_engine"] = {"frames_per_s": nfr / dt.item(), "volume_matches_single_gpu": bool(okv.item()),
                                      "note": "every level's node list evaluated in %d windows (one per GPU), values exchanged by peer-memory stores; "
                                              "at 256^3 a frame is latency-bound (one tile per SM per level), so this does not scale -- see configs3 replicas" % world}
        barrier()
        sh.unshard()
    return out if rank == 0 else None


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
