"""Every one of the 2^32 float bit patterns through the device's %g (vc_format_g) against the C library's snprintf("%g")
(tests/cpp/printf_g.c, one thread per CPU), in chunks; the host text of a chunk is made while the GPU formats it.

  python tools/format_g_exhaustive.py [--chunk-log2 26] [--log profiles/format_g_exhaustive_2p32.log]

Exits 1 at the first chunk whose texts differ, after logging the first differing value."""
import argparse
import concurrent.futures as cf
import ctypes as C
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chunk-log2", type=int, default=26)
    ap.add_argument("--log", default=None)
    a = ap.parse_args()
    from ar_voxel_project_b200.engine import format_g
    from tools.mesh_bench import gpu_info
    tmp = tempfile.mkdtemp()
    so = os.path.join(tmp, "libprintf_g.so")
    subprocess.check_call(["cc", "-O2", "-shared", "-fPIC", "-pthread", os.path.join(ROOT, "tests", "cpp", "printf_g.c"), "-o", so])
    lib = C.CDLL(so)
    lib.ref_format_g.restype = C.c_uint64
    lib.ref_format_g.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_int]
    threads = os.cpu_count() or 1
    log = open(a.log, "w") if a.log else None

    def say(msg):
        print(msg, flush=True)
        if log:
            log.write(msg + "\n")
            log.flush()

    def ref(v):
        out = np.empty(13 * len(v), np.uint8)
        n = lib.ref_format_g(v.ctypes.data, len(v), out.ctypes.data, threads)
        return out[:n].tobytes()

    chunk = 1 << a.chunk_log2
    say(f"gpu {gpu_info()}; {threads} host threads; chunks of 2^{a.chunk_log2} patterns")
    t_all = time.perf_counter()
    total_bytes = 0
    with cf.ThreadPoolExecutor(1) as pool:
        for c in range((1 << 32) // chunk):
            t0 = time.perf_counter()
            v = np.arange(c * chunk, (c + 1) * chunk, dtype=np.uint64).astype(np.uint32).view(np.float32)
            host = pool.submit(ref, v)
            got = format_g(v)
            exp = host.result()
            total_bytes += len(got)
            if got != exp:
                ga, ea = got.split(b"\n"), exp.split(b"\n")
                i = next(i for i, (x, y) in enumerate(zip(ga, ea)) if x != y)
                say(f"MISMATCH in chunk {c}: pattern 0x{c * chunk + i:08x}: device {ga[i]!r}, C library {ea[i]!r}")
                sys.exit(1)
            say(f"chunk {c:3d} [0x{c * chunk:08x}, 0x{(c + 1) * chunk - 1:08x}] equal, {len(got)} bytes, {time.perf_counter() - t0:.2f} s")
    say(f"all 2^32 patterns equal: {total_bytes} bytes of text, {time.perf_counter() - t_all:.1f} s")


if __name__ == "__main__":
    main()
