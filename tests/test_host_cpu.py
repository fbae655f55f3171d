"""CPU tests of the host-side logic: the C-ABI library loads and exports every symbol include/rendernet_b200.h
declares (no compute calls without a GPU), the reference-mirroring host functions agree with the oracle / golden
fixtures, and the batch-sharding + all-gather logic under a 2-process gloo group."""
import os
import re
import socket

import numpy as np
import pytest
import torch

from oracle import rendernet_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from rendernet_b200._lib import SIGNATURES, lib
    hdr = open(os.path.join(ROOT, "include", "rendernet_b200.h")).read()
    declared = set(re.findall(r"\b(rn_[a-z0-9_]+)\s*\(", hdr)) - {"rn_conv_desc"}
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
        assert name in SIGNATURES, f"{name} has no ctypes signature"
    assert set(SIGNATURES) == declared
    assert lib.rn_version() >= 100
    assert b"invalid" in lib.rn_error_string(-1)


def test_conv_desc_struct_matches_header_field_order():
    from rendernet_b200._lib import rn_conv_desc
    hdr = open(os.path.join(ROOT, "include", "rendernet_b200.h")).read()
    body = hdr[hdr.index("typedef struct rn_conv_desc {"):hdr.index("} rn_conv_desc;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split("{", 1)[1].split(";"):
        decl = decl.strip()
        if not decl:
            continue
        decl = re.sub(r"^(const\s+)?(int8_t|void|float|int|long long|rn_phong)\s*\**\s*", "", decl)
        names += [n.strip().lstrip("*") for n in decl.split(",")]
    assert names == [f[0] for f in rn_conv_desc._fields_]


def test_no_cpu_fallback():
    from rendernet_b200 import ops
    with pytest.raises(RuntimeError):
        ops.resample(torch.zeros(1, 4, 4, 4, 1), torch.zeros(1, 3, 4), 8, True)
    with pytest.raises(RuntimeError):
        ops.cast_to_16(torch.zeros(4))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "rendernet_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "import oracle" not in src and "from oracle" not in src, fn


def test_pose_matrices_match_oracle_and_golden(golden_dir):
    from rendernet_b200.resampling_voxel_grid import (inverse_sampling_matrix, tf_rotation_around_grid_centroid,
                                                      tf_voxel_meshgrid)
    g = np.load(os.path.join(golden_dir, "resample.npz"))
    R, S = tf_rotation_around_grid_centroid(g["chair_pose"])
    assert np.array_equal(R, g["chair_R"]) and np.array_equal(S, g["chair_S"])
    rng = np.random.default_rng(0)
    vp = np.stack([rng.uniform(0, 2 * np.pi, 8), rng.uniform(-1.4, 1.4, 8), rng.uniform(0.7, 1.4, 8)], 1).astype(np.float32)
    R, S = tf_rotation_around_grid_centroid(vp)
    Ro, So = orc.rotation_around_grid_centroid(vp)
    assert np.array_equal(R, Ro) and np.array_equal(S, So)
    assert np.array_equal(inverse_sampling_matrix(R, S, 64, 128), orc.inverse_total_matrix(Ro, So, 64, 128))
    assert np.array_equal(tf_voxel_meshgrid(4, 5, 6, True), orc.voxel_meshgrid(4, 5, 6))
    assert tf_rotation_around_grid_centroid(vp[:, :2]).shape == (8, 4, 4)       # 2-parameter form returns R only


def test_demo_helpers(golden_dir, tmp_path):
    from rendernet_b200 import Phong_shading, binvox_rw
    from rendernet_b200.RenderNet_demo import Session, compute_pose_param, load_graph
    g = np.load(os.path.join(golden_dir, "pose.npz"))
    assert np.array_equal(compute_pose_param(250.0, 60.0, 3.3), g["pose_250_60_33"])
    assert np.array_equal(Phong_shading.generate_light_pos(60.0, 250.0), g["light_60_250"])
    bv = np.load(os.path.join(golden_dir, "binvox.npz"))
    grid = np.unpackbits(bv["teapot_bits"]).reshape(64, 64, 64).astype(bool)
    flat = np.transpose(grid, (0, 2, 1)).reshape(-1).astype(np.uint8)
    rle = bytearray()
    i = 0
    while i < flat.size:
        j = i
        while j < flat.size and flat[j] == flat[i] and j - i < 255:
            j += 1
        rle += bytes([int(flat[i]), j - i])
        i = j
    p = tmp_path / "teapot.binvox"
    p.write_bytes(b"#binvox 1\ndim 64 64 64\ntranslate 0 0 0\nscale 1\ndata\n" + bytes(rle))
    with open(p, "rb") as f:
        v = binvox_rw.read_as_3d_array(f)
    assert v.data.dtype == bool and np.array_equal(v.data, grid) and int(v.data.sum()) == 27933
    with pytest.raises(KeyError):
        Session(load_graph(None)).run("encoder/nope:0", {})
    with pytest.raises(FileNotFoundError):                     # the reference's hard-coded path (RenderNet_demo.py:111)
        load_graph(str(tmp_path / "model" / "3d2d_renderer.pb"))


def test_binvox_rle_reader_rejects_bad_payloads():
    """binvox_rw.read_rle (the host half of the device decode path): header parsing and payload validation."""
    import io
    from rendernet_b200 import binvox_rw
    hdr = b"#binvox 1\ndim 2 2 2\ntranslate 0 0 0\nscale 1\ndata\n"
    dims, tr, sc, pairs = binvox_rw.read_rle(io.BytesIO(hdr + bytes([0, 3, 1, 5])))
    assert dims == [2, 2, 2] and tr == [0.0, 0.0, 0.0] and sc == 1.0 and pairs.tolist() == [[0, 3], [1, 5]]
    with pytest.raises(IOError):
        binvox_rw.read_rle(io.BytesIO(hdr + bytes([0, 3, 1])))            # odd byte count
    with pytest.raises(IOError):
        binvox_rw.read_rle(io.BytesIO(hdr + bytes([0, 3, 1, 4])))         # 7 voxels for a 2x2x2 grid
    with pytest.raises(IOError):
        binvox_rw.read_rle(io.BytesIO(b"#notbinvox\n"))


def test_variable_store_names_and_npz_spelling():
    from rendernet_b200 import tfcompat as tf
    tf.reset_default_graph(seed=3)
    with tf.variable_scope("encoder"):
        with tf.variable_scope("res1_skip"):
            with tf.variable_scope("con1_3X3"):
                w = tf.get_variable("weights", [3, 3, 3, 32, 32], initializer=tf.xavier_initializer())
                b = tf.get_variable("biases", [32], initializer=tf.constant_initializer(0.001))
    assert w._rn_name == "encoder/res1_skip/con1_3X3/weights" and tuple(w.shape) == (3, 3, 3, 32, 32)
    lim = np.sqrt(6.0 / (27 * 32 + 27 * 32))
    assert float(w.abs().max()) <= lim + 1e-7 and float(w.abs().max()) > 0.9 * lim
    assert torch.all(b == 0.001)
    tf.reset_default_graph()
    tf.load_weight_dict({"res1_skip_con1_3X3_biases": np.full(32, 0.5, np.float32),      # npz-dir spelling
                         "encoder/e_conv1/alpha:0": np.full(8, 0.25, np.float32)})       # TF spelling with :0
    with tf.variable_scope("encoder"):
        with tf.variable_scope("res1_skip"):
            with tf.variable_scope("con1_3X3"):
                b = tf.get_variable("biases", [32], initializer=tf.constant_initializer(0.001))
        with tf.variable_scope("e_conv1"):
            a = tf.get_variable("alpha", [8], initializer=tf.constant_initializer(0.0))
            with pytest.raises(ValueError):
                tf.get_variable("alpha", [9])
    assert torch.all(b == 0.5) and torch.all(a == 0.25)
    tf.reset_default_graph()


def test_shard_bounds_partition():
    from rendernet_b200.parallel import shard_bounds, turntable_poses
    for n, w in [(192, 8), (360, 8), (24, 1), (7, 3), (2, 4)]:
        cover = []
        for r in range(w):
            lo, hi = shard_bounds(n, w, r)
            assert 0 <= lo <= hi <= n
            cover += list(range(lo, hi))
        assert cover == list(range(n))
    assert shard_bounds(192, 8, 3) == (72, 96) and shard_bounds(360, 8, 7) == (315, 360)
    p = turntable_poses(72, 60.0, 3.3)
    assert p.shape == (72, 3) and abs(p[1, 0] - np.deg2rad(5.0)) < 1e-6 and abs(p[0, 1] - np.deg2rad(30)) < 1e-6


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _gloo_worker(rank, world, port, n_total, q):
    import torch.distributed as dist
    from rendernet_b200.parallel import all_gather_images, broadcast_weight_dict, shard_bounds
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    full = torch.arange(n_total * 2 * 3 * 3, dtype=torch.float32).reshape(n_total, 2, 3, 3)   # the "rendered" batch
    lo, hi = shard_bounds(n_total, world, rank)
    got = all_gather_images(full[lo:hi].clone(), n_total)
    W = {"a/weights": np.arange(6, dtype=np.float32).reshape(2, 3), "b": np.ones(4, np.float32)} if rank == 0 else None
    Wb = broadcast_weight_dict(W, src=0)
    ok = torch.equal(got, full) and np.array_equal(Wb["a/weights"], np.arange(6, dtype=np.float32).reshape(2, 3)) \
        and np.array_equal(Wb["b"], np.ones(4, np.float32))
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


@pytest.mark.parametrize("n_total", [8, 5])
def test_batch_sharding_allgather_world2_gloo(n_total):
    """world_size=2 on CPU/gloo: shard the batch, 'render', all-gather -> identical to the unsharded batch
    (even and ragged shard sizes), and the weight broadcast replicates rank 0's dict."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, n_total, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def _gloo_sharded_worker(rank, world, port, q):
    import torch.distributed as dist
    from rendernet_b200.parallel import ShardedRenderEngine
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)

    class FakeEngine:                       # the engine surface ShardedRenderEngine drives (engine.py), on CPU tensors
        B, device = 3, torch.device("cpu")

        def __init__(self):
            self.out = torch.zeros(self.B, 4, 4, 3)
            self.steps = 0

        def step_device(self):
            self.steps += 1
            self.out.copy_(torch.arange(self.B * 48, dtype=torch.float32).reshape(self.B, 4, 4, 3) + 1000.0 * rank + 0.5 * self.steps)

    ok = True
    sh = ShardedRenderEngine(FakeEngine(), gather="nccl_sync")            # the default product mode: gather between the steps
    ok = ok and sh.world == world and sh.kind == "nccl_sync"
    for step in (1, 2):
        sh.step()
        full = sh.wait()
        want = torch.cat([torch.arange(3 * 48, dtype=torch.float32).reshape(3, 4, 4, 3) + 1000.0 * r + 0.5 * step for r in range(world)])
        ok = ok and tuple(full.shape) == (world * 3, 4, 4, 3) and bool(torch.equal(full, want))
    none = ShardedRenderEngine(FakeEngine(), gather="none")
    none.step()
    ok = ok and none.wait() is none.engine.out
    try:
        ShardedRenderEngine(FakeEngine(), gather="bogus")
        ok = False
    except ValueError:
        pass
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_sharded_render_engine_world2_gloo():
    """parallel.ShardedRenderEngine (the N > 1 product API) on a 2-process gloo group with a CPU stand-in for the engine: every
    rank steps its own shard, the stream-ordered all-gather returns the whole batch in rank order, step after step."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_sharded_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def _gloo_grad_worker(rank, world, port, q):
    import zlib
    import torch.distributed as dist
    from rendernet_b200.parallel import all_reduce_gradients
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    shapes = {"enc/big/weights": (3, 3, 64, 64), "enc/big/biases": (64,), "enc/a/alpha": (8,), "enc/t/weights": (4, 4, 3, 16),
              "enc/z/weights": (5, 5, 5, 1, 8)}
    gen = lambda r: {n: torch.from_numpy(np.random.default_rng(zlib.crc32(n.encode()) % 1000 + 7 * r).standard_normal(sh).astype(np.float32))
                     for n, sh in shapes.items()}
    mine, both = gen(rank), [gen(r) for r in range(world)]
    ok = True
    for bucket in (1 << 10, 150_000, 256 << 20):            # every tensor alone / mixed / one bucket
        g = {n: t.clone() for n, t in mine.items()}
        all_reduce_gradients(g, average=True, bucket_bytes=bucket)
        for n in shapes:
            want = sum(b[n] for b in both) / world
            ok = ok and tuple(g[n].shape) == shapes[n] and bool(torch.allclose(g[n], want, atol=1e-6))
    g = {n: t.clone() for n, t in mine.items()}
    all_reduce_gradients(g, average=False)
    ok = ok and bool(torch.allclose(g["enc/a/alpha"], sum(b["enc/a/alpha"] for b in both), atol=1e-6))
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_gradient_allreduce_buckets_world2_gloo():
    """Data-parallel training's exchange step (parallel.all_reduce_gradients) on a 2-process gloo group: name-ordered flat
    buckets of three sizes give the rank average of every gradient, shapes preserved."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_grad_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): exactly one JSON line on stdout with the
    contract's keys; runs the oracle on the host cores, no GPU involved."""
    import json
    import subprocess
    import sys
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--no-b8"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "renders_per_sec" and d["unit"] == "renders/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_bench_dump_outputs_is_bounded_float32_and_samples_the_same_images(tmp_path):
    """`bench.py --dump-outputs DIR`: one float32 .npy per output, whole when it fits, else the same seeded choice of whole
    images on every run, never more than bench.DUMP_BYTES in all; the CPU reference arm refuses the option."""
    import subprocess
    import sys
    import bench
    big = np.broadcast_to(np.arange(24, dtype=np.float32)[:, None, None, None], (24, 512, 512, 3))   # 75.5 MB, image i == i
    small = np.ones((2, 3), np.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"images": big, "small": small})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["images.npy", "small.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    imgs, s = np.load(tmp_path / "a" / "images.npy"), np.load(tmp_path / "a" / "small.npy")
    assert imgs.dtype == np.float32 and s.dtype == np.float32 and np.array_equal(s, small)
    picked = imgs[:, 0, 0, 0]
    assert 10 <= len(picked) < 24 and np.all(np.diff(picked) > 0) and np.all(imgs == picked[:, None, None, None])
    assert np.array_equal(imgs, np.load(tmp_path / "b" / "images.npy"))
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "c")],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert p.returncode != 0 and "--dump-outputs" in p.stderr and not (tmp_path / "c").exists()


def test_pose_matrix_vjp_matches_finite_differences_host():
    """backward.pose_matrix_jacobian_vjp: the 3 -> 12 chain rule from dL/dMinv to dL/d(azimuth, elevation, scale) (host, float64)
    against central differences of the float32 matrix construction the forward pass uses (engine.pose_to_matrix)."""
    from rendernet_b200.backward import pose_matrix_jacobian_vjp
    from rendernet_b200.engine import pose_to_matrix
    rng = np.random.default_rng(1)
    vp = np.stack([rng.uniform(0, 6.28, 4), rng.uniform(-1.0, 1.0, 4), rng.uniform(0.8, 1.3, 4)], 1)
    dm = rng.standard_normal((4, 3, 4))
    got = pose_matrix_jacobian_vjp(vp, dm)
    assert got.shape == (4, 3)
    eps = 1e-3
    for j in range(3):
        d = np.zeros_like(vp)
        d[:, j] = eps
        fd = ((pose_to_matrix(vp + d).astype(np.float64) - pose_to_matrix(vp - d).astype(np.float64)) / (2 * eps) * dm).sum((1, 2))
        assert np.allclose(got[:, j], fd, rtol=2e-2, atol=2e-2 * np.abs(fd).max()), (j, got[:, j], fd)


def test_banded_filter_sizes_and_abi_rejections():
    """Host-only checks of the C ABI: the banded filter holds two arrangements (single CTA / CTA pair) of 9 x kblocks tiles;
    geometry the depth-folded form cannot take is rejected before any launch; exact-mode descriptors need their plane offsets."""
    from rendernet_b200._lib import lib
    assert lib.rn_conv3d_banded_bytes(32, 32, 1) == 2 * 9 * 3 * 128 * 64 * 2        # res1: 3 K blocks
    assert lib.rn_conv3d_banded_bytes(16, 32, 1) == 2 * 9 * 2 * 128 * 64 * 2        # e_conv3: 2 K blocks
    assert lib.rn_conv3d_banded_bytes(8, 16, 2) == 2 * 9 * 3 * 128 * 64 * 2         # e_conv2 (z stride 2)
    assert lib.rn_conv3d_banded_bytes(16, 16, 1) == 2 * 9 * 3 * 128 * 64 * 2        # Texture net res1
    assert lib.rn_conv3d_banded_bytes(48, 32, 1) == -1 and lib.rn_conv3d_banded_bytes(32, 32, 3) == -1
    assert lib.rn_xfold_factor(16, 512) == 4 and lib.rn_xfold_factor(32, 512) == 2 and lib.rn_xfold_factor(64, 512) == 1
    assert lib.rn_version() >= 100 and lib.rn_launch_count() >= 0


def test_variable_store_strict_and_per_engine_isolation():
    """ADVICE r1: loading a weight dict makes the store strict (a missing variable raises instead of silently falling back to a
    random initialiser; unused loaded keys are reported) and stores are independent objects (tf.use_store)."""
    from rendernet_b200 import tfcompat as tf
    a, b = tf.VariableStore(precision="exact"), tf.VariableStore(precision="fast")
    assert a.fmt == 2 and b.fmt == 0
    with tf.use_store(a):
        tf.load_weight_dict({"encoder/e_conv1/alpha": np.full(8, 0.25, np.float32), "encoder/never/used": np.zeros(1, np.float32)})
        with tf.variable_scope("encoder"):
            with tf.variable_scope("e_conv1"):
                v = tf.get_variable("alpha", [8], initializer=tf.constant_initializer(0.0))
                with pytest.raises(KeyError, match="e_conv1/biases"):
                    tf.get_variable("biases", [8], initializer=tf.constant_initializer(0.001))
                w = tf.get_variable("from_array", initializer=np.ones(3, np.float32))       # explicit arrays are always allowed
        assert torch.all(v == 0.25) and torch.all(w == 1.0) and a.unused() == ["encoder/never/used"]
        with tf.use_store(b):
            assert tf.get_store() is b and tf.compute_fmt() == 0
            with tf.variable_scope("encoder"):
                with tf.variable_scope("e_conv1"):
                    v2 = tf.get_variable("alpha", [8], initializer=tf.constant_initializer(0.0))    # b is not strict: initialiser
            assert torch.all(v2 == 0.0)
        assert tf.get_store() is a
    assert tf.get_store() is not a and "encoder/e_conv1/alpha" not in b.loaded
    with pytest.raises(ValueError):
        tf.VariableStore(precision="bf16")
