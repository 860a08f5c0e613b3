#!/usr/bin/env python
"""Developer tool: early launches (programmatic dependent launch) against the same code built with -DTRQ_NO_PDL.

    tools/build_variant.sh nopdl -DTRQ_NO_PDL
    python tools/pdl_ab.py [--runs 5] [--steps 200] [--out FILE] [-- extra bench.py arguments]

Runs bench.py (C3 and its `workloads`) alternately with the product library and with TRQ_LIB pointing at the no-PDL
build, `--runs` times each, and prints per arm and workload the median, min and max of `value` (Mrays/s), then the
median ratio. The GPU's name and power limit are read in the same call and printed first.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NOPDL = os.path.join(ROOT, "tools", "variants", "libtracer_rq_nopdl.so")


def gpu_line():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        return f"nvidia-smi unavailable: {e!r}"


def run(arm, steps, extra):
    env = dict(os.environ)
    if arm == "nopdl":
        env["TRQ_LIB"] = NOPDL
    else:
        env.pop("TRQ_LIB", None)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "10",
           "--no-cpu-baseline"] + extra
    p = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
    line = next((l for l in p.stdout.splitlines() if l.startswith("{")), None)
    if p.returncode != 0 or line is None:
        sys.stderr.write(p.stderr[-3000:])
        raise SystemExit(f"bench.py ({arm}) exited {p.returncode}")
    r = json.loads(line)
    vals = {"c3": r["value"]}
    for k, w in (r.get("workloads") or {}).items():
        if "value" in w:
            vals[k] = w["value"]
    return vals, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", help="append the raw JSON lines and the summary here")
    ap.add_argument("extra", nargs="*")
    a = ap.parse_args()
    if not os.path.exists(NOPDL):
        raise SystemExit(f"{NOPDL} missing: tools/build_variant.sh nopdl -DTRQ_NO_PDL")
    out = open(a.out, "a") if a.out else None
    head = f"# {gpu_line()}; bench.py --steps {a.steps} --no-cpu-baseline {' '.join(a.extra)}; arms alternate, {a.runs} runs each"
    print(head, flush=True)
    if out:
        out.write(head + "\n")
    res = {"pdl": [], "nopdl": []}
    for k in range(a.runs):
        for arm in (("pdl", "nopdl") if k % 2 == 0 else ("nopdl", "pdl")):
            vals, raw = run(arm, a.steps, a.extra)
            res[arm].append(vals)
            print(f"run {k} {arm:5s} " + " ".join(f"{w} {v:.1f}" for w, v in vals.items()), flush=True)
            if out:
                out.write(json.dumps({"arm": arm, "run": k, "bench": raw}) + "\n")
    lines = []
    for w in res["pdl"][0]:
        s = {}
        for arm in ("nopdl", "pdl"):
            v = [r[w] for r in res[arm] if w in r]
            s[arm] = (statistics.median(v), min(v), max(v))
        ratio = s["pdl"][0] / s["nopdl"][0]
        clear = s["pdl"][1] > s["nopdl"][2] or s["pdl"][2] < s["nopdl"][1]
        lines.append(f"{w:4s} no-PDL median {s['nopdl'][0]:8.1f} [{s['nopdl'][1]:.1f}, {s['nopdl'][2]:.1f}]   "
                     f"PDL median {s['pdl'][0]:8.1f} [{s['pdl'][1]:.1f}, {s['pdl'][2]:.1f}]   x{ratio:.4f} "
                     f"({'outside' if clear else 'inside'} both spreads)")
    print("\n".join(lines), flush=True)
    if out:
        out.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
