#!/usr/bin/env python
"""bench.py -- RenderNet forward rendering throughput on B200 (contract in the task statement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|4|5] [--precision exact|fast] [--gather nccl|peer|none]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...      # CPU restatement of the reference's TF-1 graph, host cores

Default = BASELINE.json configs[1] (and configs[2] at N = 8): a "step" is one pass of the hot path over one batch of
synthetic input: 24 random 64^3 voxel grids + poses -> resample to 128^3 -> 3-D encoder -> projection unit -> 2-D trunk ->
up-conv decoder -> 24 x 512^2 x 3 image; at N GPUs every rank renders its own 24 (weak scaling) and the output images are
all-gathered on a side stream (north_star: "NCCL all-gather only for the output image batch").
--config 4 = Texture+Normal face render B=24 (configs[3]); --config 5 = 360-frame bunny turntable sharded over the ranks
(configs[4]; a step is one sweep, the metric frames/s).

--precision: "exact" (default, the headline) = fp16 hi/lo operand pairs, 3 tensor-core products per tap: meets the 1e-3
parity bar on ANY weights (tests/test_gpu_exact.py::test_full_size_stress_weights_...); "fast" = fp16 operands, 1 product:
meets the bar for the reference's initialisers (the weights this bench uses) but not for high-gain weights.  The other
mode is timed too and reported under "other_precision".  Prints ONE JSON line (rank 0).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_RENDER = {"shader": 2.1140e12, "texture": 0.539e12}   # SURVEY.md §8(d): 1057.01 GMAC Shader RGB; 268.79+0.66 GMAC Texture
WORKLOADS = {
    2: ("renders_per_sec", "renders/s", "batch=24 random 64^3 voxels (10% occupancy), Phong shader (RenderNet_Shader) forward -> 512^2x3 fp32"),
    4: ("renders_per_sec", "renders/s", "batch=24 texture+normal face render (RenderNet_Texture_Face_Normal): random 64^3 voxels + "
                                        "199-d texture vectors -> (albedo, normal) 2 x 512^2x3 fp32"),
    5: ("frames_per_sec", "frames/s", "360-frame azimuth turntable (1 degree steps, el 60, r 3.3) of bunny.binvox, frames sharded over the ranks, "
                                      "voxel uploaded once, Phong shader forward -> 512^2x3 fp32"),
}


def synthetic_batch(B, rank=0):
    """BASELINE.md config 2 generator (SURVEY.md §8d)."""
    rng0, rng1 = np.random.default_rng(0 + 1000 * rank), np.random.default_rng(1 + 1000 * rank)
    vox = (rng0.random((B, 64, 64, 64, 1)) < 0.10).astype(np.float32)
    poses = np.stack([rng1.uniform(0, 2 * np.pi, B), (90 - rng1.uniform(10, 170, B)) * np.pi / 180,
                      3.3 / rng1.uniform(2.5, 4.5, B)], axis=1).astype(np.float32)
    return vox, poses


def synthetic_texture(B, rank=0):
    """BASELINE.md config 4: texture_in = default_rng(2).standard_normal((B,199))."""
    return np.random.default_rng(2 + 1000 * rank).standard_normal((B, 199)).astype(np.float32)


def bunny_voxel():
    bv = np.load(os.path.join(ROOT, "tests", "golden", "binvox.npz"))      # bit-packed copy of binvox/bunny.binvox
    return np.unpackbits(bv["bunny_bits"]).reshape(1, 64, 64, 64, 1).astype(np.float32)


DUMP_BYTES = 64_000_000     # --dump-outputs: total size of the .npy files, headers included


def dump_outputs(out_dir, named):
    """Writes {name: array [N, ...]} as out_dir/<name>.npy in float32, so that two builds can be compared output for
    output.  An array larger than its share of DUMP_BYTES is cut to a fixed, seeded sample of whole items along axis 0
    (sorted); which items depends only on N and the share, so equal arguments select the same items."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(named) - 4096
    for name, a in named.items():
        a = np.asarray(a, dtype=np.float32)
        per_item = a[0].nbytes
        if a.nbytes > share:
            keep = np.sort(np.random.default_rng(0).choice(a.shape[0], share // per_item, replace=False))
            print(f"dump {name}: items {keep.tolist()} of {a.shape[0]}", file=sys.stderr)
            a = a[keep]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], burst=d["bf16_tflops"], sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured")
    return dict(hbm=6650.0, burst=1590.0, sustained=1400.0, source="fallback")  # B200_PROFILING.md fallback


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self):
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self, gpu_indices):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not f[0].isdigit() or int(f[0]) not in gpu_indices:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU arm
def _use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm must still use every PHYSICAL host core (one thread per
    hyper-thread is 10x slower for oneDNN convolutions: 0.026 vs 0.30 renders/s measured on the 64-core / 128-thread box)."""
    import torch
    n = None
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
    except Exception:
        pass
    if not n:
        n = max(1, (os.cpu_count() or 2) // 2)
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    torch.set_num_threads(int(n))
    return torch.get_num_threads()


def cpu_forward_timer(config, n_renders, warm=1, batch=1):
    """Times the oracle (CPU restatement of the TF-1 graph, PyTorch-CPU oneDNN fp32) on `batch`-sized forwards of the
    config's synthetic workload; returns (seconds per forward list, threads)."""
    from oracle import rendernet_oracle as orc
    threads = _use_all_host_threads()
    if config == 4:
        W = orc.init_texture_weights(seed=0)
        vox, poses = synthetic_batch(batch)
        tex = synthetic_texture(batch)
        fn = lambda: orc.render_forward_texture(vox, tex, poses, W)            # noqa: E731
    else:
        W = orc.init_shader_weights(seed=0)
        if config == 5:
            from rendernet_b200.parallel import turntable_poses
            vox, poses = np.repeat(bunny_voxel(), batch, 0), turntable_poses(360, 60.0, 3.3)[:batch]
        else:
            vox, poses = synthetic_batch(batch)
        fn = lambda: orc.render_forward(vox, poses, W)                         # noqa: E731
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n_renders):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return ts, threads


def run_reference(args, rank, world):
    if rank != 0:
        return
    metric, unit, workload = WORKLOADS[args.config]
    ts, cores = cpu_forward_timer(args.config, args.steps, warm=max(args.warmup, 1))
    total = float(np.sum(ts))
    val = args.steps / total
    # SURVEY §8(d): also a B=8 forward (throughput form) -- one bounded sample, not part of the K timed steps
    b8 = None
    if not args.no_b8:
        t8, _ = cpu_forward_timer(args.config, 1, warm=0, batch=8)
        b8 = {"value": 8.0 / float(t8[0]), "unit": unit, "sample": "one B=8 forward after the timed steps"}
    sample = (f"{args.steps} timed B=1 forwards (one 64^3 voxel -> 512^2 image each) of the same synthetic workload on "
              f"{cores} host threads (torch.set_num_threads(physical cores), so torchrun's OMP_NUM_THREADS=1 does not apply); "
              f"oracle/rendernet_oracle.py = CPU restatement of the TF-1 graph (TensorFlow-1 itself is not installable)")
    line = {"impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "baseline_config": args.config, "step": "1 render per step (bounded CPU sample)",
                       "parallelism": "host threads"},
            "cpu_baseline": {"value": val, "unit": unit, "cores": cores, "kind": "port", "sample": sample, "b8": b8},
            "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def _file_sha(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()[:16]


def kernel_roofline(torch, ops, dev, B, cin, cout, k, precision, peaks, label):
    """Times the dominant kernel alone (CUDA events on its launch stream, 20 back-to-back launches, >= 100 MB of inputs so
    nothing survives in L2 between launches) and relates the ALGORITHMIC FLOPs of one launch to the measured burst peak."""
    fmt = 2 if precision == "exact" else 0
    x = ops.cast_to_16(torch.randn(B, 64, 64, cin, device=dev), fmt=fmt)
    w = torch.randn(k, k, cin, cout, device=dev) / float(np.sqrt(k * k * cin))
    L = ops.pack_conv("conv2d", w, torch.zeros(cout), torch.rand(cout) * 0.3, device=dev, fmt=fmt)
    y = ops.cast_to_16(torch.zeros(B, 64, 64, cout, device=dev), fmt=fmt)
    for _ in range(3):
        ops.conv2d(x, L, act="prelu", out16=y)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nl = 20
    e0.record()
    for _ in range(nl):
        ops.conv2d(x, L, act="prelu", out16=y)
    e1.record()
    torch.cuda.synchronize()
    k_ms = e0.elapsed_time(e1) / nl
    k_flop = 2.0 * B * 64 * 64 * cin * cout * k * k
    achieved = k_flop / (k_ms * 1e-3) / 1e12
    mma_per_flop = 3 if precision == "exact" else 1
    return {"kernel": label, "bound": "tensor", "achieved": achieved, "peak": peaks["burst"], "unit": "TFLOP/s",
            "frac": achieved / peaks["burst"], "peak_source": peaks["source"] + " (burst cuBLAS bf16)",
            "ms_per_launch": k_ms, "flop_per_launch": k_flop,
            "tensor_issue_tflops": achieved * mma_per_flop, "tensor_issue_frac": achieved * mma_per_flop / peaks["burst"],
            "note": ("exact mode issues 3 fp16 tensor-core products per algorithmic MAC (x_hi.w_hi + x_lo.w_hi + x_hi.w_lo): "
                     "`frac` relates ALGORITHMIC flops to the bf16 peak, `tensor_issue_frac` the issued ones"
                     if precision == "exact" else "one fp16 tensor-core product per algorithmic MAC")}


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from rendernet_b200 import ops
    from rendernet_b200.engine import RenderEngine, TextureRenderEngine
    from rendernet_b200.parallel import ShardedRenderEngine, shard_bounds, turntable_poses

    # Keep stdout clean for the single JSON line: NCCL / torchrun banners go to stderr.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = args.config
    metric, unit, workload = WORKLOADS[cfg]
    B = args.batch
    model = "texture" if cfg == 4 else "shader"
    peaks = measured_peaks()

    def build(precision, batch):
        if cfg == 4:
            return TextureRenderEngine(None, batch, use_graph=not args.no_graph, seed=0, device=f"cuda:{local_rank}", precision=precision)
        return RenderEngine(None, batch, use_graph=not args.no_graph, seed=0, device=f"cuda:{local_rank}", precision=precision)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_times(ms):
        """max over ranks (the contract) + the per-rank values (VERDICT r1: make the limiter checkable)."""
        if world == 1:
            return ms, [ms]
        t = torch.tensor([ms], device=dev)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per = [float(v.item()) for v in allt]
        return max(per), per

    # ------------------------------------------------------------------------------------------- workload set-up
    if cfg == 5:
        nframes = 360
        lo, hi = shard_bounds(nframes, world, rank)
        my_poses = turntable_poses(nframes, 60.0, 3.3)[lo:hi]
        B = (hi - lo) if (hi - lo) <= 48 else 24
        nchunk = -(-len(my_poses) // B)
        chunks = []
        for c in range(nchunk):
            p = my_poses[c * B:(c + 1) * B]
            if len(p) < B:
                p = np.concatenate([p, np.repeat(p[-1:], B - len(p), 0)])
            chunks.append(torch.from_numpy(RenderEngine.pose_to_matrix(p)))
        units_per_step_global = nframes
    else:
        vox, poses = synthetic_batch(B, rank)
        tex = synthetic_texture(B, rank) if cfg == 4 else None
        units_per_step_global = world * B

    def measure(precision, with_e2e, gather_kind, dump_dir=None):
        """-> dict(ms_step, per_rank, value, e2e..., launches) for one precision; with dump_dir, rank 0 also writes what the
        last timed step returned (dump_outputs)."""
        eng = build(precision, B)
        sh = ShardedRenderEngine(eng, gather_kind) if cfg != 5 else None
        if sh is not None and sh.peer is not None and not sh.verify_peer_against_nccl():
            raise RuntimeError("peer gather does not reproduce ncclAllGather")
        out_frames = None
        if cfg == 5:
            eng.vox.copy_(torch.from_numpy(np.repeat(bunny_voxel(), B, 0)).to(dev))          # voxel uploaded once
            pin = [c.pin_memory() for c in chunks]
            out_frames = torch.empty((nchunk * B, 512, 512, 3), device=dev, dtype=torch.float32)
            host_frames = torch.empty((nchunk * B, 512, 512, 3), dtype=torch.float32).pin_memory()
            gathered = torch.empty((world * nchunk * B, 512, 512, 3), device=dev) if world > 1 and gather_kind != "none" else None
        elif cfg == 4:
            eng.upload(vox, tex, poses)
        else:
            eng.upload(vox, poses)

        def step(e2e):
            if cfg == 5:        # one sweep: per chunk upload the poses (48 B each), replay, keep the frames
                for c in range(nchunk):
                    eng.minv.copy_(pin[c], non_blocking=True)
                    o = eng.step_device()
                    out_frames[c * B:(c + 1) * B].copy_(o)
                    if e2e:
                        host_frames[c * B:(c + 1) * B].copy_(out_frames[c * B:(c + 1) * B], non_blocking=True)
                if gathered is not None:
                    dist.all_gather_into_tensor(gathered, out_frames)
                return
            if e2e:
                tk = sh.submit(vox, tex, poses) if cfg == 4 else sh.submit(vox, poses)
                if tk > 0:
                    eng.result(tk - 1)              # the previous step's images are consumed from pinned host memory
            else:
                sh.step()

        def timed(nsteps, e2e):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(nsteps):
                step(e2e)
            if sh is not None:
                sh.wait()
            if e2e and cfg != 5:
                eng.result(eng.submitted - 1)       # last image has landed on the host
            e1.record()
            torch.cuda.synchronize()
            ms, per = rank_times(e0.elapsed_time(e1))
            barrier()
            return ms, per

        for _ in range(max(args.warmup, 3)):
            step(False)
        if with_e2e:
            for _ in range(3):                 # warm the pipelined path too (allocates its pinned / staging buffers once)
                step(True)
            if cfg != 5:
                eng.result(eng.submitted - 1)
        torch.cuda.synchronize()
        ms_total, per = timed(args.steps, False)
        if dump_dir and rank == 0:
            if cfg == 5:
                if gathered is None:
                    frames = out_frames[:len(my_poses)]
                else:                                  # every rank's block of nchunk * B frames ends in padding
                    bounds = [shard_bounds(nframes, world, r) for r in range(world)]
                    frames = torch.cat([gathered[r * nchunk * B:r * nchunk * B + hi - lo] for r, (lo, hi) in enumerate(bounds)])
                named = {"frames": frames}
            elif cfg == 4:
                named = dict(zip(("albedo", "normal"), sh.wait()))
            else:
                named = {"images": sh.wait()}
            dump_outputs(dump_dir, {k: v.cpu().numpy() for k, v in named.items()})
        phases = None
        if args.phases and sh is not None:            # where does a step's time go: graph replay vs the gather on the compute stream
            sh.timing = []
            timed(args.steps, False)
            comp, gath, period = sh.phase_times()
            sh.timing = None
            t = torch.tensor([comp, gath, period], device=dev)
            if world > 1:
                allp = [torch.zeros_like(t) for _ in range(world)]
                dist.all_gather(allp, t)
                phases = {"compute_ms_per_rank": [round(float(v[0]), 3) for v in allp], "gather_ms_per_rank": [round(float(v[1]), 3) for v in allp],
                          "period_ms_per_rank": [round(float(v[2]), 3) for v in allp]}
            else:
                phases = {"compute_ms_per_rank": [comp], "gather_ms_per_rank": [gath], "period_ms_per_rank": [period]}
        r = {"ms_step": ms_total / args.steps, "per_rank_ms": [p / args.steps for p in per], "phases": phases,
             "value": units_per_step_global * args.steps / (ms_total / 1e3),
             "launches": eng.launches_per_step * (nchunk if cfg == 5 else 1),
             "gather": sh.kind_note if sh is not None else ("NCCL all-gather of the frames" if world > 1 else "single GPU"),
             "cuda_graph": eng.graph is not None}
        if with_e2e:
            ms_e2e, per_e = timed(args.steps, True)
            r["e2e_value"] = units_per_step_global * args.steps / (ms_e2e / 1e3)
            r["e2e_per_rank_ms"] = [p / args.steps for p in per_e]
        if sh is not None:
            sh.close()
        del eng, sh
        torch.cuda.empty_cache()
        return r

    sampler = ClockSampler()
    if rank == 0:
        sampler.start()
    main_prec = args.precision
    other_prec = "fast" if main_prec == "exact" else "exact"
    try:
        M = measure(main_prec, True, args.gather, args.dump_outputs)
    finally:                                    # a failed measurement must not leave nvidia-smi sampling behind
        clocks = sampler.stop(set(range(world))) if rank == 0 else None
    O = None if args.no_other_precision else measure(other_prec, False, "none")

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel of this config, in both precisions (timed alone, inputs > L2)
    if cfg == 4:
        kshape = dict(cin=512, cout=512, k=3)
        klabel = "igemm_kernel 3x3 conv 512->512 @64x64, B=24 (Texture net res2 trunk: 21 of its launches, 75 % of its MACs)"
    else:
        kshape = dict(cin=1024, cout=1024, k=3)
        klabel = "igemm_kernel<256,cta_group::2> 3x3 conv 1024->1024 @64x64, B=24 (Shader res2 trunk: 21 of the 65 launches, 77 % of the MACs)"
    roof = kernel_roofline(torch, ops, dev, 24, precision=main_prec, peaks=peaks, label=klabel + f" [{main_prec}]", **kshape)
    roof_other = kernel_roofline(torch, ops, dev, 24, precision=other_prec, peaks=peaks, label=klabel + f" [{other_prec}]", **kshape)
    tfile = os.path.join(ROOT, "profiles", "top_kernel_traffic.json")
    roof["traffic"] = None
    if os.path.exists(tfile):
        with open(tfile) as f:
            tj = json.load(f)
        entry = tj.get(main_prec, tj if main_prec == "fast" else {})
        roof["traffic"] = entry.get("dram_bytes_per_launch")
        roof["traffic_source"] = {"file": "profiles/top_kernel_traffic.json", "sha256_16": _file_sha(tfile),
                                  "ncu_capture": entry.get("source"),
                                  "note": "dram__bytes_read.sum + dram__bytes_write.sum of this kernel from an `ncu --set full` capture "
                                          "(not measurable inside a timed run); algorithmic bytes per launch "
                                          f"{entry.get('algorithmic_bytes_per_launch')}"}
    per_flop = FLOP_PER_RENDER[model]
    step_tflops = M["value"] * per_flop / 1e12 / world
    roof["whole_step_tflops"] = step_tflops
    roof["whole_step_frac_of_sustained"] = step_tflops / peaks["sustained"]
    # projection-unit kernel (the kernel BASELINE.json's metric singles out): 1x1, K = 1024 (512 for the Texture net)
    pc = 512 if cfg == 4 else 1024
    proj = {p: kernel_roofline(torch, ops, dev, 24, cin=pc, cout=pc, k=1, precision=p, peaks=peaks,
                               label=f"projection unit 1x1 {pc}->{pc} [{p}]") for p in (main_prec, other_prec)}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        ts, cores = cpu_forward_timer(cfg, 3, warm=1)
        cpu = {"value": 3.0 / float(np.sum(ts)), "unit": unit, "cores": cores, "kind": "port",
               "sample": "3 timed B=1 forwards of the same synthetic workload on the host cores (oracle/rendernet_oracle.py, "
                         "PyTorch-CPU oneDNN fp32 restatement of the TF-1 graph), after 1 warm-up"}
    if cfg == 5:
        h2d, d2h = int(360 * 12 * 4), int(360 * 512 * 512 * 3 * 4)
        e2e_note = ("per sweep: every chunk's pose matrices go pinned host -> device (the voxel is resident: 'uploaded once'), "
                    "graph replay, every frame device -> pinned host")
    else:
        in_bytes = vox.nbytes + B * 12 * 4 + (tex.nbytes if tex is not None else 0)
        h2d, d2h = int(world * in_bytes), int(world * B * 512 * 512 * 3 * 4 * (2 if cfg == 4 else 1))
        e2e_note = ("engine.submit/result: every step stages its inputs in pinned host memory, H2D, graph replay, D2H of the images "
                    "to pinned host memory; copies of step i+-1 overlap the compute of step i (2 steps in flight); timed from the "
                    "first submit to the last image landing on the host")
    prec_note = {"exact": "fp16 hi/lo operand pairs (RN_FMT_F16X2), 3 tensor-core products per tap, fp32 accumulation; activations stored as "
                          "hi/lo pairs; matches the fp32 reference to ~1e-5 on the image for ANY weights "
                          "(tests/test_gpu_exact.py::test_full_size_stress_weights_exact_meets_bar_fast_at_its_bound)",
                 "fast": "fp16 operands and stored activations, fp32 accumulation / epilogue; meets the 1e-3 bar for the reference's "
                         "initialisers (these weights; tests/test_gpu_exact.py::test_config2_random_batch_full_size_vs_oracle[fast]) but "
                         "NOT for high-gain weights (8e-3 at gain 1.1)"}
    line = {"metric": metric, "value": M["value"], "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": M["ms_step"], "higher_is_better": True, "scaling": "strong" if cfg == 5 else "weak", "vs_baseline": None,
            "dtype": "fp16x2 (hi/lo pairs, fp32-equivalent)" if main_prec == "exact" else "fp16", "data": "synthetic",
            "config": {"workload": workload, "baseline_config": (3 if (cfg == 2 and world == 8) else cfg),
                       "global_batch": units_per_step_global, "per_gpu_batch": B,
                       "parallelism": f"dp{world} (batch sharded; output images: {M['gather']})" if world > 1 else "single GPU",
                       "weights": "reference initialisers (xavier-uniform, seeded); random-init, no checkpoint exists offline",
                       "precision": main_prec, "precision_note": prec_note[main_prec],
                       "cuda_graph": M["cuda_graph"],
                       "l2": "no explicit flush: every layer streams 200-1600 MB of activations (> 126 MB L2) per step"},
            "per_rank_ms": M["per_rank_ms"],
            "phases": M["phases"],
            "clocks": clocks,
            "e2e": {"value": M["e2e_value"], "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "per_rank_ms": M["e2e_per_rank_ms"], "note": e2e_note},
            "gpu_launches": int(M["launches"] * args.steps * 2),
            "gpu_launches_per_step": int(M["launches"]),
            "roofline": roof,
            "projection_unit": {p: {"ms_per_launch": v["ms_per_launch"], "tflops": v["achieved"], "frac_of_burst_peak": v["frac"],
                                    "tensor_issue_frac": v["tensor_issue_frac"]} for p, v in proj.items()},
            "other_precision": None if O is None else {
                "precision": other_prec, "precision_note": prec_note[other_prec], "value": O["value"], "unit": unit,
                "ms_per_step": O["ms_step"], "per_rank_ms": O["per_rank_ms"], "gather": "none (device-timed steps only)",
                "roofline": {k: roof_other[k] for k in ("kernel", "achieved", "peak", "frac", "ms_per_launch", "tensor_issue_frac")},
                "whole_step_frac_of_sustained": O["value"] * per_flop / 1e12 / world / peaks["sustained"]},
            "cpu_baseline": cpu}
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=24, help="renders per GPU per step (configs 2 and 4)")
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 4, 5],
                    help="BASELINE.json config: 2 = B=24 Shader (3 = the same at --gpus 8), 4 = Texture+Normal B=24, 5 = 360-frame turntable")
    ap.add_argument("--precision", type=str, default="exact", choices=["exact", "fast"],
                    help="headline precision mode (the other one is timed too and reported under other_precision)")
    ap.add_argument("--gather", type=str, default="nccl_sync", choices=["nccl_sync", "nccl", "peer", "none"],
                    help="N>1 output all-gather: ncclAllGather between steps on the compute stream (default), ncclAllGather overlapped "
                         "on a side stream, copy-engine P2P writes over CUDA IPC (rendernet_b200.parallel.PeerImageGather; falls back "
                         "to NCCL if IPC is unavailable), or none (ablation); see ShardedRenderEngine for the measurements")
    ap.add_argument("--phases", action="store_true", help="N>1: also record per-step device timestamps (compute vs gather) per rank")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-precision", action="store_true")
    ap.add_argument("--no-b8", action="store_true", help="reference arm: skip the extra B=8 CPU sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the headline precision's outputs of the last step as DIR/<name>.npy "
                         "(float32, at most 64 MB in all: a fixed, seeded sample of whole images when larger)")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
