#!/usr/bin/env python3
"""Runs ON THE GPU BOX: latency of one rbg_query_packed call against the batch size (what rb_align's GPU worker pays per
parsed chunk), alone and with 2 / 4 host threads calling on the same handle.  One JSON line per measurement."""
import concurrent.futures as cf
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rowbowt_b200 as rb  # noqa: E402
from rowbowt_b200 import RBG_LOCATE, RBG_NARROW_LOCS  # noqa: E402
from tools import synth  # noqa: E402

lib = rb.lib()
prefix = os.path.join(ROOT, "data", "c2", "c2")
panel = synth.make_panel(*synth.CONFIGS["c2"])
ix = rb.GpuIndex.open(prefix, sa=True, markers=False)
ix.build_ftab(10)


def pinned(nbytes, dtype):
    p = lib.rbg_host_alloc(nbytes)
    return np.frombuffer((C.c_uint8 * nbytes).from_address(p), dtype=dtype)


for n in (10_000, 53_000, 212_000, 1_000_000):
    reads = synth.make_reads(panel, n, 150, seed=3)[0]
    bases, offs = pinned(n * 150 + 64, np.uint8), pinned((n + 1) * 8, np.uint64)
    bases[:n * 150] = reads.reshape(-1)
    offs[:] = np.arange(n + 1, dtype=np.uint64) * np.uint64(150)
    packed, flags = pinned(((n * 150 + 31) // 32 + 2) * 8, np.uint64), pinned(n + 8, np.uint8)
    pb, keep = ix.pack((bases[:n * 150], offs), threads=4, out=(packed, flags))
    for mode, name in ((0, "count"), (RBG_LOCATE | RBG_NARROW_LOCS, "locate")):
        for threads in (1, 2, 4):
            reps = max(8, min(200, 4_000_000 // n))

            def loop(_):
                for _ in range(reps):
                    ix.query_raw(pb, mode)
            loop(0)
            t0 = time.perf_counter()
            with cf.ThreadPoolExecutor(threads) as ex:
                list(ex.map(loop, range(threads)))
            dt = time.perf_counter() - t0
            print(json.dumps({"kind": "call", "mode": name, "reads": n, "host_threads": threads, "calls": reps * threads,
                              "ms_per_call": dt * 1e3 / reps, "reads_per_s": n * reps * threads / dt}), flush=True)

ix.close()
