"""Row-region sharding of one image over ranks (SURVEY §8(e): the split that also cuts a single-tile image).
CPU tier: the C++ of ojb_shard.cpp / CodecBase::plan_region with world_size 2, 3 and 8 over gloo, kernels under the
SIMT emulator, against the reference's codestream and decode; seeded random geometry against the single codec.
GPU tier: the nvcc-built library with two processes on one device (callback transport staged through host memory);
tools/region_check.py runs the same configurations and two larger ones over NCCL under torchrun
(profiles/r02k_region_check_n2.json)."""
import os
import sys
import numpy as np
import pytest
import cases
import openjph_b200 as ob
from openjph_b200 import sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (parameters, writer rank).  Heights are a few slabs of 128 rows; five levels make the halo 62 (5/3) / 124 (9/7)
# rows; odd offsets move the lifting parity; the tiled case cuts every tile; the last one is too small to cut
# (ranks without rows); the tall one is for eight ranks; the DFS and the 30-bit (64-bit coefficient path) ones keep
# whole-plane transforms on every rank (general kernels) and share the block coding only.
REGION_CASES = [
    (dict(width=200, height=512, num_comps=3, bit_depth=8, num_decomps=5, reversible=True, color_transform=True), 0),
    (dict(width=333, height=700, num_comps=1, bit_depth=12, num_decomps=4, reversible=True, offset=(5, 3), block=(32, 32)), 1),
    (dict(width=256, height=640, num_comps=3, bit_depth=10, num_decomps=5, reversible=False, color_transform=True, qstep=0.004), 0),
    (dict(width=300, height=520, num_comps=3, bit_depth=8, num_decomps=3, reversible=True, subsampling=[(1, 1), (2, 2), (2, 1)],
          planar=1, prog_order="CPRL", tlm=True), 0),
    (dict(width=300, height=600, num_comps=3, bit_depth=8, num_decomps=3, reversible=True, color_transform=True,
          tile=(160, 384), tilepart_div=1), 1),
    (dict(width=96, height=100, num_comps=1, bit_depth=8, num_decomps=2, reversible=True), 0),
    (dict(width=80, height=1100, num_comps=1, bit_depth=8, num_decomps=4, reversible=True, block=(32, 32)), 0),
    (dict(width=120, height=400, num_comps=1, bit_depth=8, num_decomps=3, reversible=True, decomp="BHB", block=(32, 32)), 1),
    (dict(width=70, height=300, num_comps=1, bit_depth=30, num_decomps=3, reversible=True, block=(32, 32)), 0),
]


def _worker(rank, world, port, q, which, gpu=False):
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OJB_EMU_THREADS="2")
    import ctypes
    import torch.distributed as dist
    import refharness
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        if gpu:
            # the nvcc-built library on cuda:0, both processes on the one device; the transport callbacks stage device
            # buffers through host memory and gloo
            L = None
        else:
            import emu
            L = emu.emu_lib(build=False)
        ref = refharness.active(L)
        ok, notes = True, []

        def one_encoder(p, fr):
            # the reference's codestream; it has no writer for DFS segments (this library's extension, checked against
            # the reference's DECODER in test_part2_structures.py): there the single-process encoder is the yardstick
            if p.dfs_num_levels == 0:
                return ref.encode(p, fr)
            enc = ob.Encoder(p, ob.I32, lib=L)
            try:
                return enc.encode(fr)
            finally:
                enc.close()

        for ci in which:
            kw, writer = REGION_CASES[ci]
            writer = writer % world
            p = cases.make(kw)
            frame = cases.frame_for(p)
            sh = sharding.NativeShard(lib=L, transport="callbacks" if gpu else None)
            sh.set_partition("regions")
            sh.configure(p, ob.I32, writer=writer)
            for rep in range(2):                   # a second frame through the same objects
                fr = frame if rep == 0 else [np.ascontiguousarray(a[::-1]) for a in frame]
                # a rank reads only the rows of its slab + halo: everything else is poisoned on the other ranks
                mine = [a.copy() for a in fr]
                rows = sh.region_rows(0)
                if rows is not None and len(sharding.tile_grid(p)) == 1 and p.dy[0] == 1:
                    oy = -(-p.off_y // 1)
                    for a in mine[:1]:
                        a[:max(0, rows[0] - oy)] = -12345
                        a[max(0, rows[1] - oy):] = -12345
                cs = sh.encode(mine)
                want = one_encoder(p, fr) if rank == writer else None
                if rank == writer:
                    if p.reversible:
                        good = cs == want
                    else:
                        good = len(cs) == len(want) and cs[:cs.index(b"\xff\x90")] == want[:want.index(b"\xff\x90")]
                    if not good:
                        notes.append("case %d rep %d: encode differs (%d vs %d bytes)" % (ci, rep, len(cs), len(want)))
                    ok = ok and good
                else:
                    ok = ok and cs is None
                planes = sh.decode(want, sample_type=ob.I32, writer=writer)
                if rank == writer:
                    ref_planes, _ = ref.decode(want)
                    tol = 0 if p.reversible else 1
                    err = max(int(np.abs(a.astype(np.int64) - b).max()) for a, b in zip(planes, ref_planes))
                    if err > tol:
                        notes.append("case %d rep %d: decode off by %d" % (ci, rep, err))
                    ok = ok and err <= tol
                else:
                    ok = ok and planes is None
            # device-resident forms (under the emulator "device" memory is host memory)
            sh.upload(frame)
            addr, n = sh.encode_resident()
            want = one_encoder(p, frame) if rank == writer else None
            if rank == writer and p.reversible:
                good = (n == len(want)) if gpu else (ctypes.string_at(addr, n) == want)
                if not good:
                    notes.append("case %d: resident encode differs" % ci)
                ok = ok and good
            lens = [n]
            dist.broadcast_object_list(lens, src=writer)
            sh.decode_resident(addr, lens[0], ob.I32, writer)
            if rank == writer and not gpu:       # (device memory on a GPU: the host-buffer forms above already compared samples)
                ref_planes, _ = ref.decode(want if p.reversible else ctypes.string_at(addr, n))
                for c, rp in enumerate(ref_planes):
                    got = np.frombuffer(ctypes.string_at(sh.device_plane(c), rp.size * 4), np.int32).reshape(rp.shape)
                    good = np.abs(got.astype(np.int64) - rp).max() <= (0 if p.reversible else 1)
                    if not good:
                        notes.append("case %d: resident decode differs in component %d" % (ci, c))
                    ok = ok and good
            # an unknown partition is refused (and the object keeps the one it had)
            if (L if L is not None else sh.L).ojb_shard_set_partition(sh.h, 5) == 0:
                ok = False; notes.append("case %d: partition 5 was accepted" % ci)
            sh.close()
        q.put((rank, bool(ok), notes))
    except BaseException as e:              # the parent must hear about it instead of waiting for its timeout
        import traceback
        q.put((rank, False, ["rank %d: %r\n%s" % (rank, e, traceback.format_exc()[-1500:])]))
        raise
    finally:
        try:
            dist.destroy_process_group()
        except Exception:
            pass


def _run(world, which, timeout=600, gpu=False, worker=None):
    import multiprocessing as mp
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=worker, args=(r, world, port, q, which)) if worker is not None else
             ctx.Process(target=_worker, args=(r, world, port, q, which, gpu)) for r in range(world)]
    for pr in procs:
        pr.start()
    import queue
    import time
    res, notes = {}, []
    t0 = time.time()
    while len(res) < world and time.time() - t0 < timeout:
        try:
            r, ok, nt = q.get(timeout=2)
            res[r] = ok
            notes += nt
            if not ok:
                break                       # one rank failed: its peers would wait in a collective for ever
        except queue.Empty:
            if any(pr.exitcode not in (None, 0) for pr in procs):
                notes.append("a worker died: exit codes %s" % [pr.exitcode for pr in procs])
                break
    if len(res) < world or not all(res.values()):
        for pr in procs:
            if pr.is_alive():
                pr.kill()
    for pr in procs:
        pr.join(timeout=60)
    assert res == {r: True for r in range(world)}, notes


def test_gloo_world2_row_regions(emu_lib, ref):
    """two ranks, every case: byte-identical codestream on the writer, the reference's samples back"""
    _run(2, list(range(len(REGION_CASES))))


def test_gloo_world3_row_regions(emu_lib, ref):
    """three ranks (uneven slabs, a middle rank with a halo on both sides)"""
    _run(3, [0, 1, 2, 7, 8])


def test_gloo_world8_row_regions(emu_lib, ref):
    """eight ranks on a tall image (slabs of 128 rows, ranks that own no deep-level block) and on the 9/7 case"""
    _run(8, [6, 2])


# ---- seeded random geometry, cut fine (OJB_REGION_ALIGN=8 so that images of a hundred rows are split) -----------------
def _random_worker(rank, world, port, q, seeds):
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OJB_EMU_THREADS="2", OJB_REGION_ALIGN="8")
    import torch.distributed as dist
    import emu
    import test_random_configs as trc
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        L = emu.emu_lib(build=False)
        ok, notes, ran = True, [], 0
        for seed in seeds:
            kw = trc.random_case(seed)
            rng = np.random.default_rng(9000 + seed)
            oy = kw["offset"][1]
            kw["height"] = (kw["height"] - oy) * int(rng.integers(1, 4)) + int(rng.integers(0, 40)) + oy     # something to cut
            p = cases.make(kw)
            frame = cases.frame_for(p)
            # the single-process codec is the yardstick (itself held to the reference by test_random_configs.py); a
            # configuration it refuses -- or whose stream the decoder refuses like the reference does -- is skipped
            want, err = None, None
            if rank == 0:
                try:
                    e1 = ob.Encoder(p, ob.I32, lib=L); want = e1.encode(frame); e1.close()
                    d1 = ob.Decoder(lib=L); one = d1.decode(want, ob.I32); d1.close()
                except Exception as e:
                    err = str(e)
            flag = [err]
            dist.broadcast_object_list(flag, src=0)
            if flag[0] is not None:
                continue
            ran += 1
            sh = sharding.NativeShard(lib=L)
            sh.set_partition("regions")
            sh.configure(p, ob.I32, writer=0)
            cs = sh.encode(frame)
            planes = sh.decode(want, sample_type=ob.I32, writer=0)
            if rank == 0:
                if cs != want:
                    ok = False; notes.append("seed %d: codestream differs %r" % (seed, kw))
                elif not all(np.array_equal(a, b) for a, b in zip(planes, one)):
                    ok = False; notes.append("seed %d: samples differ %r" % (seed, kw))
            sh.close()
        if ran < len(seeds) // 2:
            ok = False; notes.append("only %d of %d configurations ran" % (ran, len(seeds)))
        q.put((rank, bool(ok), notes))
    except BaseException as e:
        import traceback
        q.put((rank, False, ["rank %d: %r\n%s" % (rank, e, traceback.format_exc()[-1500:])]))
        raise
    finally:
        try:
            dist.destroy_process_group()
        except Exception:
            pass


@pytest.mark.parametrize("world,seeds", [(2, range(0, 30)), (3, range(100, 120))], ids=["world2", "world3"])
def test_gloo_row_regions_random_geometry(world, seeds, emu_lib, ref):
    """tiles, offsets, sub-sampling, per-component coding styles, precincts, zero to five levels, 4x4 to 128x32
    code-blocks, every progression order: the regions reproduce the single encoder byte for byte and the single
    decoder sample for sample"""
    _run(world, list(seeds), worker=_random_worker)
