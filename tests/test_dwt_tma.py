"""The bulk-copy (cp.async.bulk / mbarrier) staging variant of the forward streaming DWT (OJB_DWT_TMA=1) gives the same
codestreams as the default per-lane cp.async FIFO.  The switch is read once per process, so the check runs in a child
process: emulator build in the CPU tier, the nvcc-built library on a B200 in the GPU tier."""
import os
import subprocess
import sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = r'''
import sys, os
sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
import numpy as np
import openjph_b200 as ob, images, refharness as R
lib = None
if %(emu)d:
    import emu
    lib = emu.emu_lib(build=False)
R = R.active(lib)
cases = [(1024, 200, 3, 12, dict(num_decomps=4, reversible=True, color_transform=True), ob.U16),
         (1000, 130, 1, 10, dict(num_decomps=3, reversible=True), ob.U16),
         (777, 96, 3, 16, dict(num_decomps=2, reversible=True, color_transform=True, offset=(3, 1)), ob.U16),
         (1024, 160, 3, 12, dict(num_decomps=3, reversible=False, color_transform=True, qstep=0.003), ob.U16),
         (640, 100, 3, 8, dict(num_decomps=3, reversible=True, color_transform=True), ob.I32)]
if not %(emu)d:
    cases.append((8192, 1024, 3, 12, dict(num_decomps=5, reversible=True, color_transform=True), ob.U16))
for w, h, nc, bd, kw, st in cases:
    ox, oy = kw.get("offset", (0, 0))
    fr = images.synth_frame(w - ox, h - oy, nc, bd, 11)
    p = ob.make_params(w, h, nc, bd, **kw)
    planes = [f.astype(np.uint16) for f in fr] if st == ob.U16 else fr
    cs = ob.Encoder(p, st, lib=lib).encode(planes)
    want = R.encode(p, fr)
    if kw["reversible"]:
        assert cs == want, (w, h, kw)
    else:
        assert abs(len(cs) - len(want)) <= max(4, len(want) // 1000), (w, h, kw)
        out = ob.Decoder(lib=lib).decode(cs); ref, _ = R.decode(want)
        for a, b, f in zip(out, ref, fr):          # the reference tests' tolerance: MSE within 1 %%, peak error within 1
            ma, mb = float(np.mean((a - f) ** 2.0)), float(np.mean((b - f) ** 2.0))
            assert abs(ma - mb) <= max(0.01 * mb, 0.01) and abs(int(np.abs(a - f).max()) - int(np.abs(b - f).max())) <= 1
print("tma variant ok")
'''


def _run(emu):
    env = dict(os.environ, OJB_DWT_TMA="1")
    r = subprocess.run([sys.executable, "-c", SCRIPT % dict(root=ROOT, emu=emu)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "tma variant ok" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


def test_bulk_copy_staging_emulator(emu_lib, ref):
    _run(1)


@pytest.mark.gpu
def test_bulk_copy_staging_gpu(gpu_lib, ref):
    _run(0)
