#!/usr/bin/env python
"""Cost of moving stream state: cvad_export_states / cvad_import_states of 10,000 and 65,536 v5 streams into and out of
host pageable, host pinned and device buffers, against the per-slot path (a cvad_get_state loop over 1,000 slots).

Every number is the median of `--reps` calls, each a host clock around a call that ends in a device synchronise; the
card's name and power limit are read in the same run.  Prints one JSON line."""
import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "cutter-vad_b200"))
from real_time_vad.engine import capi  # noqa: E402
from real_time_vad.engine.stream_engine import StreamEngine  # noqa: E402

REC = capi.STATE_DTYPE.itemsize


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": out[0], "power_limit": out[1]}


def timed(fn, reps):
    fn()                                         # warm-up: grows the engine's staging buffers
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return 1e3 * statistics.median(ts)


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--sizes", default="10000,65536")
    args = ap.parse_args()
    import torch
    L = capi.lib()
    res = {"metric": "state_snapshot_ms", **card(), "record_bytes": REC, "reps": args.reps, "legs": {}}
    for n in [int(x) for x in args.sizes.split(",")]:
        eng = StreamEngine("v5", max_streams=n)
        eng.reset()
        rng = np.random.default_rng(0)
        eng.step(rng.standard_normal((n, 512 * 2)).astype(np.float32) * 0.1)     # non-trivial state
        slots = np.ascontiguousarray(rng.permutation(n).astype(np.int32))
        sp = slots.ctypes.data_as(C.c_void_p)
        h = eng.handle
        pageable = np.zeros(n, capi.STATE_DTYPE)
        pin_p = L.cvad_alloc_pinned(n * REC)
        dev = torch.zeros(n * REC, dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        bufs = {"pageable": pageable.ctypes.data, "pinned": pin_p, "device": dev.data_ptr()}
        leg = {"bytes": n * REC}
        for kind, ptr in bufs.items():
            def exp(ptr=ptr):
                assert L.cvad_export_states(h, n, sp, C.c_void_p(ptr)) == 0
            def imp(ptr=ptr):
                assert L.cvad_import_states(h, n, sp, C.c_void_p(ptr)) == 0
            exp()
            leg[f"export_{kind}_ms"] = round(timed(exp, args.reps), 4)
            leg[f"import_{kind}_ms"] = round(timed(imp, args.reps), 4)
        # every buffer kind carries the same records
        pin = np.frombuffer((C.c_char * (n * REC)).from_address(pin_p), capi.STATE_DTYPE)
        assert np.array_equal(pageable.view(np.uint8), pin.view(np.uint8))
        assert np.array_equal(pageable.view(np.uint8), dev.cpu().numpy())
        L.cvad_free_pinned(C.c_void_p(pin_p))
        leg["export_pageable_GBps"] = round(n * REC / leg["export_pageable_ms"] / 1e6, 2)
        leg["import_pageable_GBps"] = round(n * REC / leg["import_pageable_ms"] / 1e6, 2)
        res["legs"][str(n)] = leg
        if n == min(int(x) for x in args.sizes.split(",")):
            hh, cc = np.zeros(128, np.float32), np.zeros(128, np.float32)
            sm, fd = np.zeros(4, np.int32), C.c_int64(0)

            def loop():
                for s in range(1000):
                    L.cvad_get_state(h, s, hh.ctypes.data, cc.ctypes.data, sm.ctypes.data, C.byref(fd))
            ms = timed(loop, max(3, args.reps // 4))
            res["get_state_loop_1000_ms"] = round(ms, 3)
            res["get_state_per_slot_us"] = round(ms, 3)            # ms per 1,000 calls == us per call
        eng.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
