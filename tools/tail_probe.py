#!/usr/bin/env python
"""Developer tool: how long the end of a trace launch is, and how much of it the next launch on the stream fills.

Needs a library built with the per-CTA timeline:
    tools/build_variant.sh tail -DTRQ_TAIL_TIMELINE                   (early launches)
    tools/build_variant.sh tailnopdl -DTRQ_TAIL_TIMELINE -DTRQ_NO_PDL (every launch waits for the previous one)
    TRQ_LIB=tools/variants/libtracer_rq_tail.so python tools/tail_probe.py [c3 c1 c4]

Each CTA of trace_packed_kernel stamps %globaltimer when it starts, when its first warp finds the ray queue exhausted and
when it exits. For every workload, four steps of bench.py's hot path run back to back, (a) as bench.py issues them,
(b) with a CUDA event recorded between steps, (c) with trq_profile_enable on. Per launch after the first:
  span      first CTA start .. last CTA exit
  tail      first "queue exhausted" stamp .. last CTA exit (the straggler tail), and its share of the step period
  gap       this launch's first CTA start - the previous launch's last exit (negative: the launches overlap)
  resident  over the tail, in tenths: % of this launch's CTAs still running / CTAs of the next launch already running
"""
import argparse
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LAUNCHES, MAX_CTAS = 8, 4096


def read_tail(lib, scene, reset):
    buf = (C.c_ulonglong * (LAUNCHES * MAX_CTAS * 3))()
    rc = lib.trq_debug_tail(scene._h, buf, C.c_int(1 if reset else 0))
    assert rc == 0, "trq_debug_tail failed"
    return np.frombuffer(buf, dtype=np.uint64).reshape(LAUNCHES, MAX_CTAS, 3).copy()


def launches(t, count):
    out = []
    for k in range(count):
        rows = t[k][t[k][:, 0] != 0]
        exh = ~rows[:, 1][rows[:, 1] != 0]                         # stored inverted (0 = this CTA never saw it)
        out.append({"start": rows[:, 0].astype(np.int64), "exit": rows[:, 2].astype(np.int64),
                    "exhausted": int(exh.min()) if exh.size else int(rows[:, 2].max())})
    return out


def report(name, mode, L):
    lines = []
    t0 = L[0]["exit"].max()
    period = (L[-1]["exit"].max() - t0) / (len(L) - 1) / 1e3
    for k in range(1, len(L)):
        a = L[k]
        nxt = L[k + 1] if k + 1 < len(L) else None
        s0, s1 = a["start"].min(), a["exit"].max()
        tail = s1 - a["exhausted"]
        gap = s0 - L[k - 1]["exit"].max()
        curve = []
        for f in np.linspace(0.0, 1.0, 11)[:-1]:
            t = a["exhausted"] + f * tail
            mine = np.mean((a["start"] <= t) & (a["exit"] > t)) * 100
            theirs = int(np.sum((nxt["start"] <= t) & (nxt["exit"] > t))) if nxt is not None else -1
            curve.append(f"{mine:.0f}/{theirs}" if nxt is not None else f"{mine:.0f}")
        lines.append(f"{name} {mode:8s} launch {k}: CTAs {a['start'].size}  span {(s1 - s0) / 1e3:8.1f} us  tail {tail / 1e3:7.1f} us "
                     f"({tail / 1e3 / period * 100:4.1f} % of the {period:.1f} us step)  gap {gap / 1e3:+7.1f} us  "
                     f"resident {' '.join(curve)}")
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=["c3", "c1", "c4"])
    ap.add_argument("--out", help="also append the lines to this file")
    a = ap.parse_args()
    import torch
    import bench
    from tracer_b200 import dist as D
    from tracer_b200._lib import lib, LIB_PATH
    if not hasattr(lib, "trq_debug_tail"):
        sys.exit(f"{LIB_PATH} has no per-CTA timeline: build it with tools/build_variant.sh <name> -DTRQ_TAIL_TIMELINE")
    lib.trq_debug_tail.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    D.init()
    torch.cuda.set_device(0)
    steps = 4
    lines = [f"# {torch.cuda.get_device_name(0)}, library {os.path.basename(LIB_PATH)}"]
    for name in a.workloads:
        w = bench.Work(name, D, 0, 0, 1)
        for _ in range(3):
            w.step()
        torch.cuda.synchronize()
        for mode in ("plain", "event", "profile"):
            read_tail(lib, w.scene, True)
            if mode == "profile":
                w.scene.profile(True)
            for _ in range(steps):
                w.step()
                if mode == "event":
                    torch.cuda.Event(enable_timing=True).record()
            torch.cuda.synchronize()
            if mode == "profile":
                w.scene.profile(False)
            lines += report(name, mode, launches(read_tail(lib, w.scene, False), steps))
        w.close()
        del w
        torch.cuda.empty_cache()
    print("\n".join(lines), flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
