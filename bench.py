#!/usr/bin/env python3
"""bench.py -- Mpixels/s encode+decode of the HTJ2K hot path.

A step = one pass of the hot path over one batch of frames: each frame is encoded to a codestream,
then that codestream is decoded back (the metric BASELINE.json names is "Mpixels/s encode+decode").
Workload at every N: synthetic 8192x8192 3-component 12-bit frames, reversible 5/3 + RCT, 5 levels,
64x64 blocks (the headline configuration), OJB_BENCH_WORKERS (default 16) frames per GPU per step, each on its
own codec object / CUDA stream so that the host phases (packet headers) and copies of one frame
overlap the kernels of another (weak scaling; frames are independent, so there is no data-path
collective -- only the final gather of the codestream sizes to rank 0).

  value : frame already resident in HBM when the timed region starts (encoder's device image
          buffer); the codestream is written to device memory and decoded FROM device memory (the
          decoder fetches only the marker segments / packet headers its host parser reads, a few
          32 KB pages per frame: ojb_dec_read_headers_device); decoded image left on the device
  e2e   : the reference-facing C-ABI frame calls with HOST buffers (pinned): H2D of the planes,
          D2H of the codestream, H2D of the codestream, D2H of the decoded planes, all timed
  --impl reference : the unmodified reference (oracle/_ref, compiled from /root/reference by
          oracle/Makefile) on the host cores the job may use (cgroup quota honoured), one process per
          core, each encoding + decoding whole 8192x8192 frames in memory with preallocated buffers

`config` is the same object in both arms (the workload); everything specific to an arm or a run is
under `detail`.  Besides the headline the GPU arm reports, under detail.configs, the other BASELINE
configurations (cfg2..cfg5), the headline through 9/7 + ICT q90 and the two extremes SURVEY 8(d) asks for
(all-zero and uniform-random frames), each with its own kernel times and frame-level roofline.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the tree may be read-only; nothing is cached in it
PROFILE_JSON = "r02_kernels.json"       # the committed ncu --set full summary the roofline's `traffic` comes from
PROFILE_FALLBACK = "r01k_kernels.json"
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W = H = 8192
NC, BD, LEVELS = 3, 12, 5
WORKLOAD = ("8192x8192x3 12-bit, reversible 5/3 + RCT, 5 levels, 64x64 code-blocks, RPCL; a step = a batch of "
            "independent frames, each encoded then decoded")
DUMP_SAMPLES = 1 << 22                  # --dump-outputs: codestream bytes sampled; half as many samples per component
CONFIG = {"workload": WORKLOAD, "l2_policy": "inputs larger than L2 (402 MB frame, 805 MB coefficients)"}


def workload_params(w=W, h=H):
    import openjph_b200 as ob
    return ob.make_params(w, h, NC, BD, num_decomps=LEVELS, reversible=True, color_transform=True)


def make_frame(w, h, seed, nc=NC, bd=BD):
    import images
    return [p.astype("uint16" if bd > 8 else "uint8") for p in images.synth_frame(w, h, nc, bd, seed)]


def usable_cpus():
    """host threads this job may really use: the affinity mask, cut down to the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    src = "affinity"
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            c = max(1, int(float(q) / float(per) + 0.5))
            if c < n:
                n, src = c, "cgroup cpu.max"
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and max(1, q // per) < n:
                n, src = max(1, q // per), "cgroup cfs quota"
        except Exception:
            pass
    return n, src


def usable_memory_bytes():
    avail = None
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                avail = int(ln.split()[1]) * 1024
    except Exception:
        pass
    try:
        m = open("/sys/fs/cgroup/memory.max").read().strip()
        if m != "max":
            cur = int(open("/sys/fs/cgroup/memory.current").read())
            left = int(m) - cur
            avail = left if avail is None else min(avail, left)
    except Exception:
        pass
    return avail


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.maxc = index, [], set(), False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0])); self.maxc = float(f[1])
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.maxc, "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------------
# CPU arms: the unmodified reference (oracle/_ref) in memory, whole frames, nothing allocated in the timed call
# ---------------------------------------------------------------------------------------------
_CPU = {}


def cpu_worker_init(frame_file):
    """per-process set-up, outside the timed region: load the reference build, the frame (int32 lines as
    ojph::codestream::exchange takes them), and pre-touch the output buffers"""
    import numpy as np
    import refharness as R
    R.lib()
    z = np.load(frame_file)
    frame = [np.ascontiguousarray(z["c%d" % c], np.int32) for c in range(NC)]
    h, w = frame[0].shape
    _CPU["frame"] = frame
    _CPU["p"] = workload_params(w, h)
    _CPU["cs"] = np.empty(w * h * NC * 2 + (1 << 20), np.uint8)
    _CPU["out"] = [np.empty((h, w), np.int32) for _ in range(NC)]
    _CPU["cs"].fill(0)                                      # every page touched before the timed region
    for a in _CPU["out"]:
        a.fill(0)


def cpu_worker(check):
    """one reference encode + decode of the frame; returns seconds (enc, dec) and the codestream size"""
    import numpy as np
    import refharness as R
    t0 = time.perf_counter(); n = R.encode_into(_CPU["p"], _CPU["frame"], _CPU["cs"]); t1 = time.perf_counter()
    R.decode_into(_CPU["cs"], n, _CPU["out"]); t2 = time.perf_counter()
    if check:
        assert all(np.array_equal(a, b) for a, b in zip(_CPU["out"], _CPU["frame"]))
    return t1 - t0, t2 - t1, n


def write_frame_file(frame):
    import numpy as np
    import tempfile
    f = tempfile.NamedTemporaryFile(prefix="ojb_bench_frame_", suffix=".npz", delete=False)
    f.close()
    np.savez(f.name, **{"c%d" % c: a for c, a in enumerate(frame)})
    return f.name


def run_cpu_reference(procs, steps, warmup, frame_file):
    """`procs` persistent processes, each one encodes + decodes one whole frame per step"""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs, initializer=cpu_worker_init, initargs=(frame_file,)) as pool:
        for i in range(max(1, warmup)):
            pool.map(cpu_worker, [i == 0] * procs, chunksize=1)
        t0 = time.perf_counter()
        per = []
        for _ in range(steps):
            per += pool.map(cpu_worker, [False] * procs, chunksize=1)
        dt = time.perf_counter() - t0
    pix = procs * steps * W * H
    te = sum(p[0] for p in per) / len(per); td = sum(p[1] for p in per) / len(per)
    return pix / dt / 1e6, dt / steps * 1e3, te, td


def bind_to_gpu_numa_node(torch, local):
    """run this rank's host threads (and first-touch its pinned buffers) on the CPUs next to its GPU:
    pinned memory on the far socket halves the PCIe rate.  Returns a note for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(local)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {w * 64 + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "%d CPUs local to GPU %s" % (len(cpus), bus)
    except Exception as e:          # no NVML / no topology information: run unbound
        return "unbound (%s)" % type(e).__name__
    return "unbound"


ENC_STAGES = ("h2d", "dwt", "ht_encode", "d2h_lengths", "host_wait", "assemble", "d2h_out", "host_ms")
DEC_STAGES = ("h2d", "host_parse", "ht_decode", "dwt_inv", "d2h_image", "_5", "_6", "host_ms")


def host_link_probe(torch, dist, world):
    """H2D + D2H of 256 MB pinned buffers at the same time on this rank's GPU, all ranks at once (behind a barrier); GB/s
    moved per rank, both directions summed.  Not part of any timed region."""
    val = -1.0
    if dist is not None:
        dist.barrier()
    try:
        n = 256 << 20
        h_in = torch.empty(n, dtype=torch.uint8, pin_memory=True); h_out = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        h_in.zero_()
        d_a = torch.empty(n, dtype=torch.uint8, device="cuda"); d_b = torch.zeros(n, dtype=torch.uint8, device="cuda")
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

        def go():
            with torch.cuda.stream(s1):
                d_a.copy_(h_in, non_blocking=True)
            with torch.cuda.stream(s2):
                h_out.copy_(d_b, non_blocking=True)
        go(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(6):
            go()
        torch.cuda.synchronize()
        val = 2 * 6 * n / (time.perf_counter() - t0) / 1e9
    except Exception:
        val = -1.0
    if dist is None:
        return [round(val, 1)]
    try:
        t = torch.tensor([val], device="cuda", dtype=torch.float64)
        g = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(g, t)
        return [round(float(x.item()), 1) for x in g]
    except Exception:
        return [round(val, 1)]


def sharded_block(a, rank, world, L, ob, np, torch, dist, C, _lib, peak):
    """Strong scaling of ONE image over the ranks: every rank passes the whole image (host, pinned), codes its tiles,
    tile-part bytes / decoded samples go device to device over NCCL to rank 0, which delivers the codestream / the
    planes to host memory.  Timed: encode + decode per frame, barrier + synchronize on both sides, max over ranks,
    the gathers inside the timed region.  Checked outside it: the codestream equals the one a single encoder on
    rank 0 produces (itself byte-identical to the reference, tests/), and the round trip."""
    from openjph_b200 import sharding
    steps = max(2, min(a.steps, 5))
    out = {"transport": "NCCL send/recv + allgather inside libojph_b200.so (ojb_shard.cpp); tiles: tile t on rank t % N; row regions: "
                        "slab g of every tile-component on rank g", "entries": []}

    def timed_loop(fn, n):
        dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n * 1e3

    def one(name, params, frame, lossless, partition=0):
        st = ob.U8 if frame[0].dtype == np.uint8 else ob.U16
        pin = [torch.empty(f.shape, dtype=torch.uint8 if f.dtype == np.uint8 else torch.uint16, pin_memory=True) for f in frame]
        for t, f in zip(pin, frame):
            t.numpy()[:] = f
        nc = len(frame)
        planes = (C.c_void_p * nc)(*[t.data_ptr() for t in pin])
        in_bytes = sum(f.nbytes for f in frame)
        cap = in_bytes * 2 + (1 << 20)
        cs_pin = torch.empty(cap if rank == 0 else 16, dtype=torch.uint8, pin_memory=True)
        out_pin = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in pin] if rank == 0 else None
        outs = (C.c_void_p * nc)(*[t.data_ptr() for t in out_pin]) if rank == 0 else None
        sh = sharding.NativeShard()
        n = C.c_uint64(); fi = _lib.FrameInfo()

        def ck(rc):
            if rc != 0:
                raise RuntimeError(L.ojb_shard_last_error().decode())

        if partition:
            ck(L.ojb_shard_set_partition(sh.h, partition))
        ck(L.ojb_shard_enc_configure(sh.h, C.byref(params), st, 0))

        def enc():
            ck(L.ojb_shard_enc_encode(sh.h, planes, None, cs_pin.data_ptr(), cs_pin.numel(), C.byref(n)))

        def dec():
            ck(L.ojb_shard_dec_decode(sh.h, cs_pin.data_ptr(), cs_len, st, 0, outs, None, C.byref(fi)))

        enc()
        cs_len = int(n.value)
        dec()
        e = {"workload": name, "ranks": world, "partition": "row regions" if partition else "tiles"}
        if partition:
            lo, hi = C.c_uint32(), C.c_uint32()
            rows = [0, 0]
            if L.ojb_shard_region_rows(sh.h, 0, C.byref(lo), C.byref(hi)):
                rows = [int(lo.value), int(hi.value)]
            rt = torch.tensor(rows, dtype=torch.int64, device="cuda")
            allr = [torch.zeros_like(rt) for _ in range(world)]
            dist.all_gather(allr, rt)
            e["input_rows_per_rank"] = [[int(x[0]), int(x[1])] for x in allr]      # slab + halo each rank reads
        # the same image on one GPU (rank 0 alone): reference point of the strong scaling, and the byte-identity check
        one_gpu_ms = None
        if rank == 0:
            enc1 = L.ojb_enc_create(); dec1 = L.ojb_dec_create()
            try:
                if L.ojb_enc_configure(enc1, C.byref(params), st) != 0:
                    raise RuntimeError(L.ojb_last_error().decode())
                cs1 = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
                o1 = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in pin]
                o1p = (C.c_void_p * nc)(*[t.data_ptr() for t in o1])
                n1 = C.c_uint64()

                def single():
                    assert L.ojb_enc_encode_frame(enc1, planes, None, cs1.data_ptr(), cap, C.byref(n1)) == 0, L.ojb_last_error()
                    assert L.ojb_dec_read_headers(dec1, cs1.data_ptr(), n1.value, st, C.byref(fi)) == 0, L.ojb_last_error()
                    assert L.ojb_dec_decode_frame(dec1, o1p, None) == 0, L.ojb_last_error()
                single(); single()
                torch.cuda.synchronize(); t0 = time.perf_counter()
                for _ in range(steps):
                    single()
                torch.cuda.synchronize(); one_gpu_ms = (time.perf_counter() - t0) / steps * 1e3
                e["codestream_identical_to_one_gpu"] = bool(n1.value == cs_len and torch.equal(cs1[:cs_len], cs_pin[:cs_len]))
                if lossless:
                    e["round_trip_lossless"] = bool(all(np.array_equal(o.numpy(), f) for o, f in zip(out_pin, frame)))
                else:
                    e["max_abs_diff_vs_one_gpu_decode"] = int(max(np.abs(o.numpy().astype(np.int64) - q.numpy().astype(np.int64)).max() for o, q in zip(out_pin, o1)))
            finally:
                L.ojb_enc_destroy(enc1); L.ojb_dec_destroy(dec1)
        for _ in range(2):
            enc(); dec()
        ms_enc = timed_loop(enc, steps)
        ms_dec = timed_loop(dec, steps)
        ms_both = timed_loop(lambda: (enc(), dec()), steps)
        # device-resident form: tiles already in each rank's HBM, codestream gathered into rank 0's HBM and decoded from
        # there, decoded image gathered into rank 0's HBM -- no PCIe traffic besides headers, so what is timed is the
        # sharded compute + the NCCL exchange (the host-buffer form above is bound by rank 0's PCIe link either way)
        ck(L.ojb_shard_enc_upload(sh.h, planes, None))
        nres = C.c_uint64()
        lens_t = torch.zeros(1, dtype=torch.int64, device="cuda")

        def res():
            ck(L.ojb_shard_enc_encode_resident(sh.h, C.byref(nres)))
            ck(L.ojb_shard_dec_decode_resident(sh.h, L.ojb_shard_device_codestream(sh.h), cs_len, st, 0, C.byref(fi)))
        res(); res()
        ms_res = timed_loop(res, steps)
        # where one frame's time goes on the writer (CUDA events inside the library; not part of the timed loops)
        tm = (C.c_float * 2)()
        ck(L.ojb_shard_enc_encode_resident(sh.h, C.byref(nres))); L.ojb_shard_timings(sh.h, tm); split_e = (float(tm[0]), float(tm[1]))
        ck(L.ojb_shard_dec_decode_resident(sh.h, L.ojb_shard_device_codestream(sh.h), cs_len, st, 0, C.byref(fi))); L.ojb_shard_timings(sh.h, tm)
        split_d = (float(tm[0]), float(tm[1]))
        one_gpu_res_ms = None
        if rank == 0:
            enc1 = L.ojb_enc_create(); dec1 = L.ojb_dec_create()
            try:
                assert L.ojb_enc_configure(enc1, C.byref(params), st) == 0, L.ojb_last_error()
                assert L.ojb_enc_upload_frame(enc1, planes, None) == 0, L.ojb_last_error()
                csd = torch.empty(cap, dtype=torch.uint8, device="cuda")
                n1 = C.c_uint64()

                def single_res():
                    assert L.ojb_enc_encode_resident(enc1, csd.data_ptr(), cap, C.byref(n1), 1) == 0, L.ojb_last_error()
                    assert L.ojb_dec_read_headers_device(dec1, csd.data_ptr(), n1.value, st, C.byref(fi)) == 0, L.ojb_last_error()
                    assert L.ojb_dec_decode_resident(dec1) == 0, L.ojb_last_error()
                single_res(); single_res()
                torch.cuda.synchronize(); t0 = time.perf_counter()
                for _ in range(steps):
                    single_res()
                torch.cuda.synchronize(); one_gpu_res_ms = (time.perf_counter() - t0) / steps * 1e3
            finally:
                L.ojb_enc_destroy(enc1); L.ojb_dec_destroy(dec1)
        dist.barrier()
        if rank == 0:
            pix = frame[0].shape[0] * frame[0].shape[1]
            e.update({"host_buffers": {"ms_per_frame_encode": round(ms_enc, 3), "ms_per_frame_decode": round(ms_dec, 3), "ms_per_frame": round(ms_both, 3),
                                       "Mpixels_per_s": round(pix / ms_both / 1e3, 1), "one_gpu_ms_per_frame": round(one_gpu_ms, 3),
                                       "time_vs_one_gpu": round(ms_both / one_gpu_ms, 3),
                                       "note": "pinned host buffers on rank 0: every rank uploads its own tiles, rank 0's PCIe link carries the whole "
                                               "codestream and the whole decoded image, so this form cannot scale"},
                      "device_resident": {"ms_per_frame": round(ms_res, 3), "Mpixels_per_s": round(pix / ms_res / 1e3, 1),
                                          "one_gpu_ms_per_frame": round(one_gpu_res_ms, 3), "time_vs_one_gpu": round(ms_res / one_gpu_res_ms, 3),
                                          "writer_split_ms": {"encode_own_share": round(split_e[0], 3), "encode_exchange_headers_layout": round(split_e[1], 3),
                                                              "decode_broadcast_parse_own_share": round(split_d[0], 3), "decode_gather": round(split_d[1], 3)},
                                          "note": "one frame at a time (latency, not a stream): encode + NCCL gather of tile-parts + NCCL broadcast + decode + "
                                                  "NCCL gather of samples, against the same two calls on one GPU"},
                      "codestream_bytes": cs_len})
            out["entries"].append(e)
        sh.close()

    tile_w = {2: 4096, 4: 4096, 8: 2048}.get(world, 4096)
    one("cfg4: 8192x8192x3 16-bit, reversible 5/3 + RCT, 4 tiles of 4096x4096, 5 levels",
        ob.make_params(W, H, 3, 16, num_decomps=5, reversible=True, color_transform=True, tile=(4096, 4096)), make_frame(W, H, 9, 3, 16), True)
    one("headline frame as %d tiles of %dx4096 (12-bit, 5/3 + RCT, 5 levels)" % ((W // tile_w) * 2, tile_w),
        ob.make_params(W, H, NC, BD, num_decomps=LEVELS, reversible=True, color_transform=True, tile=(tile_w, 4096)), make_frame(W, H, 1234), True)

    # the headline frame as it is -- ONE tile -- cut into N row regions (SURVEY 8(e)): input halo, no mid-pipeline exchange,
    # code-block bytes gathered to rank 0 which writes the packet headers; byte-identical to the one-GPU codestream
    if os.environ.get("OJB_BENCH_REGIONS", "1") != "0":
        one("headline frame, single tile, as %d row regions (12-bit, 5/3 + RCT, 5 levels)" % world,
            ob.make_params(W, H, NC, BD, num_decomps=LEVELS, reversible=True, color_transform=True), make_frame(W, H, 1234), True, partition=1)

    # cfg5: a batch of 64 independent 4K frames, frame f on rank f % N, codestreams gathered to rank 0 over NCCL
    try:
        nfr = 64
        p5 = ob.make_params(3840, 2160, 3, 10, num_decomps=5, reversible=False, color_transform=True)
        fr = make_frame(3840, 2160, 10, 3, 10)
        pin = [torch.empty(f.shape, dtype=torch.uint16, pin_memory=True) for f in fr]
        for t, f in zip(pin, fr):
            t.numpy()[:] = f
        planes = (C.c_void_p * 3)(*[t.data_ptr() for t in pin])
        mine = [f for f in range(nfr) if f % world == rank]
        NW5 = 4
        encs = []
        for _ in range(NW5):
            e_ = L.ojb_enc_create()
            assert L.ojb_enc_configure(e_, C.byref(p5), ob.U16) == 0, L.ojb_last_error()
            encs.append(e_)
        per = 3840 * 2160 * 3 * 2
        slot = (per * 6 // 10 + 4095) & ~4095                   # the default step size gives ~6 bits / sample on this frame
        dev = torch.empty(len(mine) * slot + (1 << 20), dtype=torch.uint8, device="cuda")
        gat = torch.empty((nfr * slot + (1 << 20)) if rank == 0 else 16, dtype=torch.uint8, device="cuda")
        host = torch.empty(gat.numel(), dtype=torch.uint8, pin_memory=True)
        sh = sharding.NativeShard()
        offs = (C.c_uint64 * (world + 1))()
        from concurrent.futures import ThreadPoolExecutor
        tp = ThreadPoolExecutor(NW5)

        def batch():
            lens = [0] * len(mine)

            def work(k):
                n_ = C.c_uint64()
                for i in range(k, len(mine), NW5):
                    assert L.ojb_enc_upload_frame(encs[k], planes, None) == 0, L.ojb_last_error()
                    assert L.ojb_enc_encode_resident(encs[k], dev.data_ptr() + i * slot, slot, C.byref(n_), 1) == 0, L.ojb_last_error()
                    lens[i] = int(n_.value)
            list(tp.map(work, range(NW5)))
            # pack this rank's codestreams back to back, then one variable-length gather to rank 0 and one D2H
            pos = 0
            for i, ln_ in enumerate(lens):
                if pos != i * slot:
                    dev[pos:pos + ln_].copy_(dev[i * slot:i * slot + ln_].clone())
                pos += ln_
            torch.cuda.synchronize()
            assert L.ojb_shard_gatherv(sh.h, dev.data_ptr(), pos, 0, gat.data_ptr(), gat.numel(), offs) == 0, L.ojb_shard_last_error()
            if rank == 0:
                host[:offs[world]].copy_(gat[:offs[world]], non_blocking=True)
                torch.cuda.synchronize()
            return pos
        batch()
        ms = timed_loop(batch, 2)
        if rank == 0:
            out["entries"].append({"workload": "cfg5: batch of 64 independent 3840x2160x3 10-bit frames, irreversible 9/7 + ICT, frame f on rank f % N, "
                                               "codestreams gathered to rank 0 (NCCL) and copied to host; encode only", "ranks": world,
                                   "ms_per_batch": round(ms, 2), "Mpixels_per_s_encode": round(nfr * 3840 * 2160 / ms / 1e3, 1),
                                   "gathered_bytes": int(offs[world])})
        for e_ in encs:
            L.ojb_enc_destroy(e_)
        sh.close()
    except Exception as ex:
        if rank == 0:
            out["entries"].append({"workload": "cfg5", "error": str(ex)[:300]})
    return out if rank == 0 else None


def main():
    # the contract is ONE JSON line on stdout: keep the real stdout for it and send everything libraries
    # print at C level (e.g. NCCL's version banner) to stderr
    out = os.fdopen(os.dup(1), "w")
    sys.stdout.flush()
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last device-resident step of the headline returned as DIR/*.npy: "
                         "the codestream's length, its first 64 KiB and a fixed sample of its bytes, and a fixed sample of the "
                         "decoded samples of every component (positions drawn with numpy's default_rng(0); about 40 MB)")
    a = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = dict(CONFIG)

    if a.impl == "reference":
        if rank != 0:
            return
        import refharness as R
        if not R.available():
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref was not built (needs /root/reference at build time)"}), file=out); out.flush()
            return
        cores, src = usable_cpus()
        procs = int(os.environ.get("OJB_BENCH_CPU_PROCS", "0")) or cores
        mem = usable_memory_bytes()
        per_proc = W * H * NC * (4 + 4 + 2) + (512 << 20)          # int32 frame + int32 output + codestream + slack
        if mem is not None:
            procs = max(1, min(procs, int(mem * 0.6) // per_proc))
        frame_file = write_frame_file(make_frame(W, H, 1234))
        try:
            v, ms, te, td = run_cpu_reference(procs, max(1, a.steps), max(0, min(a.warmup, 1)), frame_file)
        finally:
            os.unlink(frame_file)
        sample = ("%d processes (%s: %d usable CPUs of %d in the affinity mask) x one whole 8192x8192x3 12-bit frame per step, in-memory "
                  "files, buffers preallocated; per process encode %.2f s decode %.2f s; ISA level %d" % (
                      procs, src, cores, len(os.sched_getaffinity(0)), te, td, R.lib().ojr_cpu_ext_level()))
        print(json.dumps({"impl": "reference", "metric": "Mpixels/s encode+decode", "value": v, "unit": "Mpixels/s",
                          "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
                          "data": "synthetic", "config": cfg, "detail": {"frames_per_step": procs},
                          "cpu_baseline": {"value": v, "unit": "Mpixels/s", "cores": procs, "kind": "reference", "sample": sample},
                          "e2e": {"value": v, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), file=out)
        out.flush()
        return

    import numpy as np
    import torch
    import openjph_b200 as ob
    from openjph_b200 import _lib
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = _lib.lib()
    assert L.ojb_set_device(local) == 0, L.ojb_last_error()
    torch.cuda.set_device(local)
    affinity = bind_to_gpu_numa_node(torch, local)      # before any pinned allocation (first touch)
    NW = int(os.environ.get("OJB_BENCH_WORKERS", "16"))     # frames in flight per GPU (one codec pair each; 12 -> 16 still buys ~3 %, gpurun_out value_probe; profiles/README.md)

    def ck(rc):
        if rc != 0:
            raise RuntimeError(L.ojb_last_error().decode())

    # frames in flight through HOST buffers (`e2e`): the PCIe link saturates earlier than the SMs, and every such frame
    # pins 0.8 GB of host memory -- fewer of them (value_probe: e2e peaks at 8)
    NE = min(NW, int(os.environ.get("OJB_BENCH_E2E_WORKERS", "8")))

    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max(NW, 32))

    class Workload:
        """one configuration: a frame (list of uint8/uint16 planes), parameters, `n` codec pairs"""
        def __init__(self, params, frame, n):
            self.p = params
            self.frame = frame
            self.st = ob.U8 if frame[0].dtype == np.uint8 else ob.U16
            self.nc = len(frame)
            self.pix = frame[0].shape[0] * frame[0].shape[1]
            self.in_bytes = sum(f.nbytes for f in frame)
            self.pin = [torch.empty(f.shape, dtype=torch.uint8 if f.dtype == np.uint8 else torch.uint16, pin_memory=True) for f in frame]
            for t, f in zip(self.pin, frame):
                t.numpy()[:] = f
            self.planes = (C.c_void_p * self.nc)(*[t.data_ptr() for t in self.pin])
            self.cs_cap = self.in_bytes * 2 + (1 << 20)
            self.ne = min(n, NE)
            self.workers = [Worker(self, i < self.ne) for i in range(n)]

        def close(self):
            for w in self.workers:
                L.ojb_enc_destroy(w.enc); L.ojb_dec_destroy(w.dec)
            self.workers = []

    class Worker:
        def __init__(self, wl, host=True):
            self.wl = wl
            self.host = host             # has pinned host buffers: takes part in the e2e leg
            self.enc = L.ojb_enc_create(); self.dec = L.ojb_dec_create()
            ck(L.ojb_enc_configure(self.enc, C.byref(wl.p), wl.st))
            if host:
                self.out_pin = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in wl.pin]
                self.outs = (C.c_void_p * wl.nc)(*[t.data_ptr() for t in self.out_pin])
                self.cs_pin = torch.empty(wl.cs_cap, dtype=torch.uint8, pin_memory=True)
            self.cs_dev = torch.empty(wl.cs_cap, dtype=torch.uint8, device="cuda")
            self.n = C.c_uint64(); self.fi = _lib.FrameInfo(); self.cs_len = 0

        def e2e(self):
            wl = self.wl
            ck(L.ojb_enc_encode_frame(self.enc, wl.planes, None, self.cs_pin.data_ptr(), wl.cs_cap, C.byref(self.n)))
            ck(L.ojb_dec_read_headers(self.dec, self.cs_pin.data_ptr(), self.n.value, wl.st, C.byref(self.fi)))
            ck(L.ojb_dec_decode_frame(self.dec, self.outs, None))

        def resident(self):
            ck(L.ojb_enc_encode_resident(self.enc, self.cs_dev.data_ptr(), self.wl.cs_cap, C.byref(self.n), 1))
            ck(L.ojb_dec_read_headers_device(self.dec, self.cs_dev.data_ptr(), self.n.value, self.wl.st, C.byref(self.fi)))
            ck(L.ojb_dec_decode_resident(self.dec))

    def timed(workers, fn_name, steps):
        """`steps` steps of len(workers) frames each; with several workers every worker streams its own
        `steps` frames back to back (no per-step barrier: frames of one worker overlap the other
        workers' copies and host phases, as in a continuous stream)"""
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if len(workers) == 1:
            for _ in range(steps):
                getattr(workers[0], fn_name)()
        else:
            def loop(w):
                f = getattr(w, fn_name)
                for _ in range(steps):
                    f()
            list(pool.map(loop, workers))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); dt = float(t.item())
        return dt

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6650 GB/s"

    class DeviceArray:
        """a view of device memory the library owns, for torch.as_tensor"""
        def __init__(self, ptr, n, typestr):
            self.__cuda_array_interface__ = {"data": (int(ptr), False), "shape": (n,), "typestr": typestr, "version": 2}

    def resident_outputs(w):
        """what one device-resident step hands its caller: the codestream in device memory and the decoded planes in the
        decoder's image buffer, sampled at seeded positions so that two builds compare output for output"""
        wl, n = w.wl, int(w.n.value)
        rng = np.random.default_rng(0)
        pos = torch.from_numpy(np.sort(rng.integers(0, n, DUMP_SAMPLES))).cuda()
        out = {"codestream_length": np.array([n], np.float64),
               "codestream_head": w.cs_dev[:min(n, 1 << 16)].float().cpu().numpy(),
               "codestream_sample": w.cs_dev[pos].float().cpu().numpy()}
        h, wd = wl.frame[0].shape
        pix = torch.from_numpy(np.sort(rng.integers(0, h * wd, DUMP_SAMPLES // 2))).cuda()
        typestr = "|u1" if wl.st == ob.U8 else "<i2"
        for c in range(wl.nc):
            plane = torch.as_tensor(DeviceArray(L.ojb_dec_device_plane(w.dec, c), h * wd, typestr), device="cuda")
            v = plane[pix].to(torch.int32)
            out["decoded_c%d" % c] = (v & 0xFFFF if typestr == "<i2" else v).float().cpu().numpy()
        torch.cuda.synchronize()
        return out

    def measure(wl, steps, warmup, lossless, e2e=True, dump=False):
        """correctness of what is timed, then: serial pass (per-stage CUDA-event times), all workers in flight
        resident (`value`), all workers in flight through host buffers (`e2e`)"""
        ws = wl.workers
        wh = [w for w in ws if w.host]
        for w in ws:
            if w.host:
                w.e2e()
                w.cs_len = w.n.value
                if lossless:
                    for a_, b_ in zip(w.out_pin, wl.frame):
                        assert np.array_equal(a_.numpy(), b_), "round trip is not lossless"
            ck(L.ojb_enc_upload_frame(w.enc, wl.planes, None))
        for _ in range(max(3, warmup)):
            list(pool.map(lambda w: w.resident(), ws))
        if lossless:                        # the device-resident path decodes the same samples
            pl = (C.c_void_p * wl.nc)(*[t.data_ptr() for t in ws[0].out_pin])
            for t in ws[0].out_pin:
                t.zero_()
            ck(L.ojb_dec_decode_frame(ws[0].dec, pl, None))
            for a_, b_ in zip(ws[0].out_pin, wl.frame):
                assert np.array_equal(a_.numpy(), b_), "device-resident round trip is not lossless"
        te = (C.c_float * 8)(); td = (C.c_float * 8)()
        dt_serial = timed(ws[:1], "resident", steps)
        L.ojb_enc_timings(ws[0].enc, te); L.ojb_dec_timings(ws[0].dec, td)
        dt_res = timed(ws, "resident", steps)
        outputs = resident_outputs(ws[0]) if dump else None
        r = {"outputs": outputs, "dt_serial": dt_serial, "dt_res": dt_res, "dt_e2e": None, "te": list(te), "td": list(td), "te2": None, "td2": None,
             "cs_len": int(ws[0].cs_len), "mirror_bytes": int(L.ojb_dec_mirror_bytes(ws[0].dec))}
        if e2e:
            for _ in range(max(1, min(warmup, 2))):
                list(pool.map(lambda w: w.e2e(), wh))
            r["dt_e2e"] = timed(wh, "e2e", steps)
            te2 = (C.c_float * 8)(); td2 = (C.c_float * 8)()
            L.ojb_enc_timings(ws[0].enc, te2); L.ojb_dec_timings(ws[0].dec, td2)
            r["te2"], r["td2"] = list(te2), list(td2)
        return r

    def frame_roofline(wl, r):
        """SURVEY 8(d): A = S_in + S_out per frame and direction; the two-pass budget A2 = A + 2 * 4 bytes per sample"""
        se = dict(zip(ENC_STAGES, r["te"])); sd = dict(zip(DEC_STAGES, r["td"]))
        samples = sum(f.size for f in wl.frame)
        A = wl.in_bytes + r["cs_len"]; A2 = A + 8 * samples
        t_enc = (se["dwt"] + se["ht_encode"] + se["assemble"]) * 1e-3
        t_dec = (sd["ht_decode"] + sd["dwt_inv"]) * 1e-3
        return {"A_bytes": A, "A2_bytes": A2, "encode_kernels_ms": round(t_enc * 1e3, 3), "decode_kernels_ms": round(t_dec * 1e3, 3),
                "encode_frac_A": round(A / t_enc / 1e9 / peak, 4), "encode_frac_A2": round(A2 / t_enc / 1e9 / peak, 4),
                "decode_frac_A": round(A / t_dec / 1e9 / peak, 4), "decode_frac_A2": round(A2 / t_dec / 1e9 / peak, 4),
                "encode_Mpix_s_device": round(wl.pix / t_enc / 1e6, 1), "decode_Mpix_s_device": round(wl.pix / t_dec / 1e6, 1)}

    def summarize(name, wl, r, steps, note=None):
        n = len(wl.workers)
        d = {"workload": name, "frames_in_flight": n,
             "Mpixels_per_s": round(wl.pix * n * a.gpus * steps / r["dt_res"] / 1e6, 1),
             "serial_ms_per_frame": round(r["dt_serial"] / steps * 1e3, 3), "codestream_bytes": r["cs_len"],
             "bits_per_sample": round(8.0 * r["cs_len"] / sum(f.size for f in wl.frame), 3),
             "stages_encode_ms": {k: round(float(v), 4) for k, v in zip(ENC_STAGES, r["te"])},
             "stages_decode_ms": {k: round(float(v), 4) for k, v in zip(DEC_STAGES, r["td"]) if not k.startswith("_")},
             "roofline_frame": frame_roofline(wl, r)}
        if r["dt_e2e"]:
            d["e2e_Mpixels_per_s"] = round(wl.pix * wl.ne * a.gpus * steps / r["dt_e2e"] / 1e6, 1)
            d["e2e_frames_in_flight"] = wl.ne
        if note:
            d["note"] = note
        return d

    # ---- headline --------------------------------------------------------------------------
    p = workload_params()
    frame = make_frame(W, H, 1234 + rank)
    head = Workload(p, frame, NW)
    sampler = ClockSampler(local); sampler.start()
    r = measure(head, a.steps, a.warmup, True, dump=bool(a.dump_outputs) and rank == 0)
    if r["outputs"]:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in r["outputs"].items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)
    sampler.stop_flag = True; sampler.join(timeout=2)
    cs_len = r["cs_len"]
    enc, dec = head.workers[0].enc, head.workers[0].dec
    launches = int(L.ojb_enc_kernel_launches(enc) + L.ojb_dec_kernel_launches(dec))
    head.close()

    # ---- the other configurations and the extremes (reported under detail.configs; not part of `value`) ----
    configs = []
    if os.environ.get("OJB_BENCH_EXTRAS", "1") != "0":
        xs = max(2, min(a.steps, 3))
        rng = np.random.default_rng(99 + rank)

        def run_cfg(name, params, frm, nworkers, lossless, note=None, e2e=True):
            try:
                wl = Workload(params, frm, nworkers)
                try:
                    # small frames: enough steps for a timed region of ~0.2 s (a few milliseconds of work measure the
                    # scheduler, not the kernels); the entry says how many
                    ws_ = wl.workers
                    for w in ws_:
                        if w.host:
                            w.e2e()
                        ck(L.ojb_enc_upload_frame(w.enc, wl.planes, None))
                    list(pool.map(lambda w: w.resident(), ws_))
                    dt1 = timed(ws_, "resident", 1)
                    steps_c = int(min(200, max(xs, np.ceil(0.2 / max(dt1, 1e-4)))))
                    d_ = summarize(name, wl, measure(wl, steps_c, 3, lossless, e2e), steps_c, note)
                    d_["steps"] = steps_c
                    configs.append(d_)
                finally:
                    wl.close()
            except Exception as e:      # the headline numbers stand on their own
                configs.append({"workload": name, "error": str(e)[:300]})

        run_cfg("headline frame, irreversible 9/7 + ICT, Qfactor 90",
                ob.make_params(W, H, NC, BD, num_decomps=LEVELS, reversible=False, color_transform=True, qfactor=90), frame, 4, False)
        run_cfg("extreme: all-zero 8192x8192x3 12-bit frame (best case for the block coders), 5/3 + RCT", p,
                [np.zeros((H, W), np.uint16) for _ in range(NC)], 2, True, e2e=False)
        run_cfg("extreme: uniform-random full-range 8192x8192x3 12-bit frame (worst case, ~12 bits/sample), 5/3 + RCT", p,
                [rng.integers(0, 1 << BD, (H, W), dtype=np.uint16) for _ in range(NC)], 2, True, e2e=False)
        run_cfg("cfg2: 1920x1080 RGB 8-bit, reversible 5/3 + RCT, 5 levels",
                ob.make_params(1920, 1080, 3, 8, num_decomps=5, reversible=True, color_transform=True), make_frame(1920, 1080, 7, 3, 8), 8, True,
                note="small frames: one frame is 1 519 code-blocks = 48 warps; more than 8 frames in flight LOWER the rate (32: 4.4 Gpixel/s): about 45 launches per frame, the stream is bound by the launch rate of the process")
        run_cfg("cfg3: 4096x4096x3 12-bit, irreversible 9/7 + ICT, Qfactor 90, 6 levels",
                ob.make_params(4096, 4096, 3, 12, num_decomps=6, reversible=False, color_transform=True, qfactor=90), make_frame(4096, 4096, 8, 3, 12), 8, False)
        run_cfg("cfg4 on one GPU: 8192x8192x3 16-bit, reversible 5/3 + RCT, 4 tiles of 4096x4096, 5 levels",
                ob.make_params(W, H, 3, 16, num_decomps=5, reversible=True, color_transform=True, tile=(4096, 4096)), make_frame(W, H, 9, 3, 16), 4, True,
                note="the 4-tiles-over-4-GPUs form of this configuration is the `sharded` entry of a --gpus 4 run")
        run_cfg("cfg5: 3840x2160x3 10-bit frames, irreversible 9/7 + ICT (qstep default), 5 levels; batch of 64 / N GPUs, 8 in flight",
                ob.make_params(3840, 2160, 3, 10, num_decomps=5, reversible=False, color_transform=True), make_frame(3840, 2160, 10, 3, 10), 8, False)

    # ---- one image over the N GPUs (SURVEY 8(e)): tiles sharded over ranks below the C-ABI, NCCL gather to rank 0 ----
    sharded = None
    if dist is not None and os.environ.get("OJB_BENCH_SHARDED", "1") != "0":
        try:
            sharded = sharded_block(a, rank, world, L, ob, np, torch, dist, C, _lib, peak)
        except Exception as e:
            sharded = {"error": str(e)[:300]}

    # what the host side of every GPU's link delivers while ALL ranks copy at once (pinned memory, H2D and D2H together):
    # `e2e` moves 631 MB per frame and direction, and GPUs that share a socket share its memory / IO bandwidth
    link = host_link_probe(torch, dist, world)

    # final gather of the per-rank codestream sizes (the only collective on the frame-parallel path)
    sizes = [cs_len]
    if dist is not None:
        t = torch.tensor([cs_len], device="cuda", dtype=torch.int64)
        g = [torch.zeros_like(t) for _ in range(world)] if rank == 0 else None
        dist.gather(t, g, dst=0)
        if rank == 0:
            sizes = [int(x.item()) for x in g]
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    pix = W * H * a.gpus * NW
    value = pix * a.steps / r["dt_res"] / 1e6
    e2e = W * H * a.gpus * head.ne * a.steps / r["dt_e2e"] / 1e6
    stage_e = {k: round(float(v), 4) for k, v in zip(ENC_STAGES, r["te"])}
    stage_d = {k: round(float(v), 4) for k, v in zip(DEC_STAGES, r["td"]) if not k.startswith("_")}
    e2e_e = {k: round(float(v), 3) for k, v in zip(ENC_STAGES, r["te2"])}
    e2e_d = {k: round(float(v), 3) for k, v in zip(DEC_STAGES, r["td2"]) if not k.startswith("_")}
    # dominant kernel = the slowest device stage of the resident step
    samples = W * H * NC
    cand = {"ht_encode": (stage_e["ht_encode"], 4 * samples + cs_len), "ht_decode": (stage_d["ht_decode"], 4 * samples + cs_len),
            "dwt_fwd": (stage_e["dwt"], 2 * samples + 4 * samples * 4 // 3 + 4 * samples // 3),
            "dwt_inv": (stage_d["dwt_inv"], 2 * samples + 4 * samples * 4 // 3 + 4 * samples // 3)}
    dom = max(cand, key=lambda k: cand[k][0])
    ach = cand[dom][1] / (cand[dom][0] * 1e-3) / 1e9 if cand[dom][0] > 0 else 0.0
    # DRAM bytes of the same kernel(s) from the committed ncu --set full capture (profiles/)
    traffic = None; traffic_src = None
    for pj in (PROFILE_JSON, PROFILE_FALLBACK):
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", pj)))
            keys = {"ht_encode": ["ht_encode_fast", "ht_encode_serial", "ht_encode"],
                    "ht_decode": ["ht_decode_fast", "ht_decode_serial", "ht_dec_fill", "ht_dec_step1", "ht_dec_step2"],
                    "dwt_fwd": ["dwt_fwd"], "dwt_inv": ["dwt_inv"]}[dom]
            traffic = sum(int(prof[k]["traffic_bytes"]) for k in keys if k in prof)
            traffic_src = "profiles/" + pj
            break
        except Exception:
            pass
    roof = {"bound": "hbm", "kernel": dom, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
            "frac": round(ach / peak, 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": cand[dom][1], "ms_per_launch": cand[dom][0],
            "note": "entropy-coding kernels are instruction-issue / ALU-pipe bound (DRAM traffic ~= algorithmic bytes); see profiles/README.md",
            "frame": frame_roofline(head, r)}
    detail = {"frames_per_step": NW * a.gpus, "frames_in_flight_per_gpu": NW, "e2e_frames_in_flight_per_gpu": head.ne, "host_affinity": affinity,
              "serial_ms_per_frame": round(r["dt_serial"] / a.steps * 1e3, 3),
              "serial_Mpixels_per_s": round(W * H * a.steps / r["dt_serial"] / 1e6, 1),
              "stages_encode_ms": stage_e, "stages_decode_ms": stage_d,
              "e2e_stages_encode_ms": e2e_e, "e2e_stages_decode_ms": e2e_d, "codestream_bytes": sizes,
              "resident_decode_header_fetch_bytes": r["mirror_bytes"],
              "pipeline_hbm_frac": round(((2 * samples + cs_len) * 2 * NW) / (r["dt_res"] / a.steps) / 1e9 / peak, 4),
              "host_link_duplex_GBps_per_rank": link,
              "configs": configs, "sharded": sharded}
    res = {"metric": "Mpixels/s encode+decode", "value": value, "unit": "Mpixels/s", "n_gpus": a.gpus, "steps": a.steps,
           "warmup": a.warmup, "ms_per_step": r["dt_res"] / a.steps * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": cfg, "detail": detail,
           "value_note": "device-resident: frame in HBM, codestream written to and decoded from HBM; the encoder produces packet "
                         "headers and markers on the device (only the length returns to the host); the decoder's host parser "
                         "fetches only marker segments / packet headers (%d bytes of the %d-byte codestream per frame, inside the "
                         "timed region)" % (r["mirror_bytes"], cs_len),
           "clocks": sampler.summary(),
           "e2e": {"value": e2e, "unit": "Mpixels/s", "h2d_bytes_per_step": (W * H * NC * 2 + cs_len) * a.gpus * head.ne,
                   "d2h_bytes_per_step": (W * H * NC * 2 + cs_len) * a.gpus * head.ne, "ms_per_step": r["dt_e2e"] / a.steps * 1e3,
                   "frames_per_step": head.ne * a.gpus},
           "gpu_launches": launches * a.steps * NW,
           "roofline": roof}
    if not a.no_cpu_baseline:
        import refharness as R
        if R.available():
            ff = write_frame_file(frame)
            try:
                cpu_worker_init(ff)
            finally:
                os.unlink(ff)
            te_ = td_ = 0.0
            reps = 2
            for _ in range(reps):
                e_, d_, _n = cpu_worker(False); te_ += e_; td_ += d_
            v1 = reps * W * H / (te_ + td_) / 1e6
            res["cpu_baseline"] = {"value": v1, "unit": "Mpixels/s", "cores": 1, "kind": "reference",
                                   "sample": "%d x one whole 8192x8192x3 12-bit frame, 1 thread (the library's native mode), in-memory, "
                                             "buffers preallocated; encode %.1f Mpix/s decode %.1f Mpix/s; ISA level %d" % (
                                                 reps, reps * W * H / te_ / 1e6, reps * W * H / td_ / 1e6, R.lib().ojr_cpu_ext_level())}
    print(json.dumps(res), file=out); out.flush()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
