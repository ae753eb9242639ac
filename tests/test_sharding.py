"""Tile sharding across ranks (SURVEY §8(e)).  CPU tier: host logic + the N>1 path over gloo with
world_size 2, kernels under the SIMT emulator; GPU tier: the same over NCCL in tools/gpu_multi.sh
(tests/test_gpu_parity.py covers the single-process form on a real device)."""
import os
import sys
import numpy as np
import pytest
import cases
import openjph_b200 as ob
from openjph_b200 import sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TILED = dict(width=300, height=200, num_comps=3, bit_depth=8, num_decomps=3, reversible=True, color_transform=True,
             tile=(128, 128), tlm=True)
TILED_OFF = dict(width=300, height=200, num_comps=1, bit_depth=8, num_decomps=3, reversible=True, tile=(128, 100),
                 offset=(7, 5), tile_offset=(3, 2), tilepart_div=1)
TILED_SUB = dict(width=200, height=150, num_comps=3, bit_depth=8, num_decomps=2, reversible=True, tile=(96, 64),
                 subsampling=[(1, 1), (2, 2), (2, 2)], planar=1)


def test_tile_grid_and_split_roundtrip(ref):
    p = cases.make(TILED)
    grid = sharding.tile_grid(p)
    assert len(grid) == 6 and grid[5]["x0"] == 256 and grid[5]["x1"] == 300 and grid[5]["y1"] == 200
    frame = cases.frame_for(p)
    cs = ref.encode(p, frame)
    header, parts = sharding.split_codestream(cs)
    assert [t for t, _ in parts] == list(range(6))
    assert header + b"".join(b for _, b in parts) + b"\xff\xd9" == cs
    geo = sharding.siz_params(header)
    assert (geo.width, geo.height, geo.tile_w, geo.tile_h, geo.num_comps) == (300, 200, 128, 128, 3)


@pytest.mark.parametrize("kw", [TILED, TILED_OFF, TILED_SUB], ids=["rgb_tlm", "offsets_tileparts", "sub420"])
def test_sharded_encode_is_the_reference_codestream(kw, emu_lib, ref):
    """tiles encoded one by one as one-tile images and re-assembled == the reference's codestream"""
    p = cases.make(kw)
    frame = cases.frame_for(p)
    want = ref.encode(p, frame)
    grid = sharding.tile_grid(p)
    parts = {}
    for r in range(2):          # two "ranks", sequentially
        parts.update(sharding.encode_tiles(p, frame, [grid[t] for t in sharding.my_tiles(len(grid), r, 2)], ob.I32, emu_lib))
    got = sharding.assemble(p, parts, lib=emu_lib)
    assert got == want
    geo, grid2, tiles = sharding.decode_tiles(want, range(len(grid)), ob.I32, emu_lib)
    out = sharding.paste_tiles(geo, grid2, tiles)
    for a, b in zip(out, frame):
        assert np.array_equal(a, b)


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OJB_EMU_THREADS="2")
    import torch.distributed as dist
    import emu, refharness
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        L = emu.emu_lib(build=False)
        ref = refharness.active(L)
        p = cases.make(TILED)
        frame = cases.frame_for(p)
        cs = sharding.encode_sharded(p, frame, ob.I32, lib=L)
        ok = True
        if rank == 0:
            ok = cs == ref.encode(p, frame)
        # decode side: every rank holds the stream, planes gathered on rank 0
        blob = [cs]
        dist.broadcast_object_list(blob, src=0)
        planes = sharding.decode_sharded(blob[0], ob.I32, lib=L)
        if rank == 0:
            ok = ok and all(np.array_equal(a, b) for a, b in zip(planes, frame))
        else:
            ok = ok and cs is None and planes is None
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_gloo_world2_sharded_encode_decode(emu_lib, ref):
    import multiprocessing as mp
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    res = {}
    for _ in range(2):
        r, ok = q.get(timeout=240)
        res[r] = ok
    for pr in procs:
        pr.join(timeout=60)
        assert pr.exitcode == 0
    assert res == {0: True, 1: True}


# ---- the native path (ojb_shard.cpp): tile masks below the C-ABI, transport behind callbacks --------------------
def _native_worker(rank, world, port, q):
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OJB_EMU_THREADS="2")
    import torch.distributed as dist
    import emu, refharness
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        L = emu.emu_lib(build=False)
        ref = refharness.active(L)
        ok = True
        for kw, writer in ((TILED, 0), (TILED_OFF, 1), (TILED_SUB, 0),
                           (dict(width=256, height=192, num_comps=3, bit_depth=12, num_decomps=3, reversible=False, color_transform=True,
                                 qstep=0.002, tile=(128, 96)), 0)):
            p = cases.make(kw)
            frame = cases.frame_for(p)
            sh = sharding.NativeShard(lib=L)
            sh.configure(p, ob.I32, writer=writer)
            for rep in range(2):                   # a second frame through the same objects
                fr = frame if rep == 0 else [np.ascontiguousarray(a[::-1]) for a in frame]
                cs = sh.encode(fr)
                want = ref.encode(p, fr) if rank == writer else None
                if rank == writer:
                    if p.reversible:
                        ok = ok and cs == want
                    else:
                        ok = ok and len(cs) == len(want) and cs[:cs.index(b"\xff\x90")] == want[:want.index(b"\xff\x90")]
                else:
                    ok = ok and cs is None
                planes = sh.decode(want, sample_type=ob.I32, writer=writer)
                if rank == writer:
                    ref_planes, _ = ref.decode(want)
                    tol = 0 if p.reversible else 1
                    ok = ok and all(np.abs(a.astype(np.int64) - b).max() <= tol for a, b in zip(planes, ref_planes))
                else:
                    ok = ok and planes is None
            # device-resident forms (under the emulator "device" memory is host memory: read it back directly)
            import ctypes
            sh.upload(frame)
            addr, n = sh.encode_resident()
            want = ref.encode(p, frame) if rank == writer else None
            if rank == writer and p.reversible:
                ok = ok and ctypes.string_at(addr, n) == want
            lens = [n]
            dist.broadcast_object_list(lens, src=writer)
            fi = sh.decode_resident(addr, lens[0], ob.I32, writer)
            if rank == writer:
                ref_planes, _ = ref.decode(want if p.reversible else ctypes.string_at(addr, n))
                for c, rp in enumerate(ref_planes):
                    got = np.frombuffer(ctypes.string_at(sh.device_plane(c), rp.size * 4), np.int32).reshape(rp.shape)
                    ok = ok and np.abs(got.astype(np.int64) - rp).max() <= (0 if p.reversible else 1)
            sh.close()
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_gloo_world2_native_shard(emu_lib, ref):
    """world_size 2 over gloo: the C++ sharded encoder / decoder (tile masks, size allgather, tile-part and sample
    gathers through the transport callbacks) against the reference's codestream and decode"""
    import multiprocessing as mp
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_native_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    res = {}
    for _ in range(2):
        r, ok = q.get(timeout=300)
        res[r] = ok
    for pr in procs:
        pr.join(timeout=60)
        assert pr.exitcode == 0
    assert res == {0: True, 1: True}
