"""world_size-2 gloo tests of the multi-GPU host logic (frame sharding, reference-frame broadcast)."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from kvazaar_b200 import dist as kd


def test_shard_frames_partition():
    for world in (1, 2, 4, 8):
        seen = sorted(i for r in range(world) for i in kd.shard_frames(37, r, world))
        assert seen == list(range(37))
        assert all(kd.owner_of(i, world) == r for r in range(world) for i in kd.shard_frames(37, r, world))


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        frames = 5
        mine = kd.shard_frames(frames, rank, world)
        ok = True
        for f in range(frames):
            buf = torch.full((64 * 64 * 3 // 2,), f + 1, dtype=torch.uint8) if f in mine else torch.zeros(64 * 64 * 3 // 2, dtype=torch.uint8)
            kd.broadcast_reference_frame(buf, f, world)
            ok &= bool((buf == f + 1).all())
        sizes = kd.gather_result_sizes(100 + rank)
        ok &= sizes == [100 + r for r in range(world)]
        out[rank] = ok
    finally:
        dist.destroy_process_group()


def test_broadcast_reference_frame_gloo_world2():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    assert dict(out) == {0: True, 1: True}
    assert np.all([out[0], out[1]])


def test_tile_grid_matches_reference_rule():
    """Uniform tile split (encoder.c:383-391): boundary i = i * size_in_ctus / count, in CTUs."""
    xs, ys = kd.tile_grid(7680, 4320, 4, 2)
    assert xs == [0, 1920, 3840, 5760, 7680] and ys == [0, 2176, 4320]          # 120 x 68 CTUs -> 30-CTU columns, 34-CTU rows
    xs, ys = kd.tile_grid(1920, 1080, 4, 2)
    assert xs == [0, 448, 960, 1408, 1920] and ys == [0, 512, 1080]              # 30 x 17 CTUs -> 7,8,7,8 columns; 8,9 rows
    assert [kd.tile_of_rank(r, 4, 2) for r in range(8)] == [(c, r) for r in range(2) for c in range(4)]


def _tile_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        W, H, cols, rows = 256, 192, 2, 1
        rng = np.random.default_rng(3)
        full = torch.from_numpy(rng.integers(0, 256, W * H * 3 // 2, dtype=np.uint8))
        xs, ys = kd.tile_grid(W, H, cols, rows)
        # every rank starts with only its own tile filled in
        mine = torch.zeros_like(full)
        tx, ty = kd.tile_of_rank(rank, cols, rows)
        for off, pw, ph, sub in ((0, W, H, 1), (W * H, W // 2, H // 2, 2), (W * H * 5 // 4, W // 2, H // 2, 2)):
            x0, x1, y0, y1 = xs[tx] // sub, xs[tx + 1] // sub, ys[ty] // sub, ys[ty + 1] // sub
            mine[off:off + pw * ph].view(ph, pw)[y0:y1, x0:x1] = full[off:off + pw * ph].view(ph, pw)[y0:y1, x0:x1]
        kd.allgather_tile_reconstructions(mine, W, H, cols, rows)
        out[rank] = bool(torch.equal(mine, full))
    finally:
        dist.destroy_process_group()


def test_allgather_tile_reconstructions_gloo_world2():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_tile_worker, args=(2, port, out), nprocs=2, join=True)
    assert dict(out) == {0: True, 1: True}


# ---- the CTU search driver's N > 1 path: pictures sharded over ranks (all-intra pictures are independent, no data-path
# collective), each rank encodes its shard with its own provider, times are max-reduced: gloo, two ranks, host provider
def _ctu_shard_worker(rank, world, port, clip, out_dir, out):
    import hashlib
    import subprocess
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        ref_dir = os.path.join(root, "oracle", "_ref")
        w, h, frames = 128, 64, 6
        fsz = w * h * 3 // 2
        data = np.fromfile(clip, dtype=np.uint8).reshape(frames, fsz)
        mine = kd.shard_frames(frames, rank, world)
        shard = os.path.join(out_dir, f"shard{rank}.yuv")
        data[mine].tofile(shard)
        res = {}
        for name, binary, env in (("ref", "kvz_stream_bench_ref", {}),
                                  ("ctu", "kvz_stream_bench_ctu", {"KVZ_CTU_PROVIDER": os.path.join(root, "tests", "hostsim", "libkvzctu_hostsim.so")})):
            e = dict(os.environ)
            e.pop("KVZ_CTU_PROVIDER", None)
            e.update(env)
            o = os.path.join(out_dir, f"{name}{rank}.hevc")
            r = subprocess.run([os.path.join(ref_dir, binary), shard, f"{w}x{h}", o, str(len(mine)), "1", "0", "0", "preset=medium", "qp=27", "period=1"],
                               env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
            assert r.returncode == 0, r.stderr[-800:]
            res[name] = hashlib.sha256(open(o, "rb").read()).hexdigest()
        same = res["ref"] == res["ctu"]
        # the bench's reduction: whole-job frames over the slowest rank's time
        t = torch.tensor([1.0 + rank], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        n = torch.tensor([float(len(mine))], dtype=torch.float64)
        dist.all_reduce(n, op=dist.ReduceOp.SUM)
        out[rank] = (same, float(t.item()), float(n.item()))
    finally:
        dist.destroy_process_group()


def test_ctu_driver_pictures_shard_over_ranks_gloo_world2(tmp_path):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for f in ("kvz_stream_bench_ref", "kvz_stream_bench_ctu"):
        if not os.path.exists(os.path.join(root, "oracle", "_ref", f)):
            import pytest
            pytest.skip("oracle/_ref stream bench hosts missing")
    from test_ctu_driver import _hostsim
    _hostsim()                                                  # builds the host library if it is missing
    sys.path.insert(0, os.path.join(root, "tools"))
    from synth_yuv import synth_frame
    clip = str(tmp_path / "c.yuv")
    with open(clip, "wb") as fh:
        for i in range(6):
            fh.write(synth_frame(128, 64, 1234, i).tobytes())
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_ctu_shard_worker, args=(2, port, clip, str(tmp_path), out), nprocs=2, join=True)
    assert out[0][0] and out[1][0], "a rank's shard differs from the reference's bitstream of the same pictures"
    assert out[0][1] == out[1][1] == 2.0 and out[0][2] == out[1][2] == 6.0


# ---- the exchange measurement bench.py attaches to its N > 1 lines (kvazaar_b200/dist.py: measure_exchanges), on gloo:
# 10-bit tiles travel as bytes (neither NCCL nor gloo has a 16-bit integer type), every rank must end up with every tile
def _exchange_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        r = kd.measure_exchanges(torch.device("cpu"), iters=2, tile_res=(512, 256), frame_res=(256, 128))
        out[rank] = (r["tile_allgather"]["verified"], r["reference_broadcast"]["verified"], r["tile_allgather"]["tiles"], r["ranks"])
    finally:
        dist.destroy_process_group()


def test_measure_exchanges_gloo_world2_and_4():
    for world, tiles in ((2, "2x1"), (4, "2x2")):
        s = socket.socket()
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
        s.close()
        mgr = mp.Manager()
        out = mgr.dict()
        mp.spawn(_exchange_worker, args=(world, port, out), nprocs=world, join=True)
        assert dict(out) == {r: (True, True, tiles, world) for r in range(world)}
