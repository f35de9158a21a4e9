"""Timeline of the mapping stage's end-of-sweep map update inside the streaming pipeline (bench.py's "value" arm).

    python tools/map_update_timeline.py [--out DIR] [--warmup 5] [--steps 20] [--windows 3] [--split-update]

DIR defaults to map_update_timeline/ under the system's temporary directory.

Runs the bench workload (hdl64_1m, bench.py's sweeps and map) through Pipeline.submit / collect with the sweeps in
HBM, and reports per timed sweep and as medians:
  (a) the update span: first to last device operation of the update (kernels and memsets on the streams that run the
      update's own kernels), its operation count and summed kernel time, and the span of every one of those streams;
  (b) the launch latency of the update: end of the sweep's last map_iterate_kernel to the update's first operation;
  (c) how long the next begin_sweep's single readback waits (LOAM_B200_TRACE's "[begin_sweep] ... wait");
  (d) n_ins (stack points inserted) and n_raw (raw seed points of the cubes in view) per kind, and how often
      S = n_ins + n_raw exceeds CS_MAX_N = 65536 (the single-cluster limit).
(c) and (d) come from windows without the profiler; (a) and (b) from one extra window under torch.profiler with CUDA
activities, whose chrome trace is written to DIR/timeline.pt.trace.json.  The card name and power limit go into
DIR/summary.json next to the figures.  --split-update runs the multi-launch update chain for every sweep
(LOAM_B200_SPLIT_MAP_UPDATE=1), the form sweeps above the single-cluster limit take.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
os.environ["LOAM_B200_TRACE"] = "1"  # read once by the library: set before it is loaded
if "--split-update" in sys.argv:
    os.environ["LOAM_B200_SPLIT_MAP_UPDATE"] = "1"  # read when a context is created

CS_MAX_N = 65536
# kernels that only the map update launches; the streams they run on are the update's streams
UPDATE_ONLY = ("store_insert_kernel", "store_front_cluster", "store_raw_select", "store_valid_by_slot", "store_voxel_merge",
               "runs_below_kernel", "store_live_count", "store_merge_kernel", "store_stats_kernel", "store_index_kernel")
BURST_GAP_US = 60.0  # operations of one update follow each other closely; consecutive sweeps' updates are >= 200 us apart
BEGIN_RE = re.compile(r"\[begin_sweep\].*wait (\d+) us, n_ins (\d+) (\d+), n_raw (\d+) (\d+)")


def card_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info["power_limit_sm_mhz_max_sm_mhz"] = q.stdout.strip()
    except Exception as e:  # noqa: BLE001
        info["power_limit_sm_mhz_max_sm_mhz"] = f"unavailable: {e!r}"
    return info


def run_window(api, work, warmup, steps, profiler=None):
    """One fresh pipeline, warmup + steps sweeps through submit / collect (bench.py's streaming device-input loop)."""
    corner, surf, sweeps, d_sweeps = work
    pipe = api.Pipeline()
    pipe.seed_map(corner, surf)
    poses = []

    def run(lo, hi):
        got = 0
        for i in range(lo, hi):
            pipe.submit(ring_sizes=sweeps[i][1], device_ptr=d_sweeps[i].data_ptr())
            r = pipe.collect(wait=False)
            if r is not None:
                poses.append(r)
                got += 1
        while got < hi - lo:
            poses.append(pipe.collect(wait=True))
            got += 1
        pipe.sync()

    run(0, warmup)
    pipe.stage_seconds(reset=True)
    if profiler is not None:
        profiler.start()
    run(warmup, warmup + steps)
    if profiler is not None:
        profiler.stop()
    ss = pipe.stage_seconds()
    del pipe
    return poses, ss


def med(xs):
    return round(statistics.median(xs), 2) if xs else None


def base_name(e):
    """kernel name without return type, namespace, template arguments and parameters; "memset" for memsets"""
    if e["cat"] != "kernel":
        return "memset"
    return e["name"].split("(")[0].split("<")[0].replace("void ", "").split("::")[-1]


def analyse_trace(path):
    ev = json.load(open(path))["traceEvents"]
    gpu = [e for e in ev if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memset")]
    upd_streams = {e["args"].get("stream") for e in gpu if e["cat"] == "kernel" and base_name(e).startswith(UPDATE_ONLY)}
    ops = sorted((e for e in gpu if e["args"].get("stream") in upd_streams), key=lambda e: e["ts"])
    iters = sorted((e for e in gpu if e["cat"] == "kernel" and "map_iterate_kernel" in e["name"]), key=lambda e: e["ts"])
    bursts, cur = [], []
    for e in ops:
        if cur and e["ts"] - max(o["ts"] + o["dur"] for o in cur) > BURST_GAP_US:
            bursts.append(cur)
            cur = []
        cur.append(e)
    if cur:
        bursts.append(cur)
    rows = []
    for b in bursts:
        t0 = b[0]["ts"]
        t1 = max(o["ts"] + o["dur"] for o in b)
        prev_iter_end = max((k["ts"] + k["dur"] for k in iters if k["ts"] + k["dur"] <= t0), default=None)
        per_stream = {}
        for o in b:
            s = per_stream.setdefault(o["args"].get("stream"), [o["ts"], o["ts"] + o["dur"], 0])
            s[0] = min(s[0], o["ts"])
            s[1] = max(s[1], o["ts"] + o["dur"])
            s[2] += 1
        names = {}
        for o in b:
            nm = base_name(o)
            names[nm] = names.get(nm, 0.0) + o["dur"]
        rows.append({"span_us": round(t1 - t0, 2), "ops": len(b),
                     "kernels": sum(1 for o in b if o["cat"] == "kernel"),
                     "kernel_us": round(sum(o["dur"] for o in b if o["cat"] == "kernel"), 2),
                     "launch_latency_us": round(t0 - prev_iter_end, 2) if prev_iter_end is not None else None,
                     "stream_spans_us": sorted((round(v[1] - v[0], 2) for v in per_stream.values()), reverse=True),
                     "stream_ops": sorted((v[2] for v in per_stream.values()), reverse=True),
                     "kernel_us_by_name": {k: round(v, 2) for k, v in sorted(names.items(), key=lambda kv: -kv[1])}})
    return rows, len(upd_streams)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "map_update_timeline"))
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--windows", type=int, default=3, help="windows without the profiler for (c) and (d)")
    ap.add_argument("--split-update", action="store_true", help="the multi-launch update chain for every sweep")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)

    import torch
    from bench import make_workload
    from loam_velodyne_b200 import api
    _, corner, surf, sweeps = make_workload("hdl64_1m", args.warmup + args.steps)
    d_sweeps = [torch.from_numpy(p).to("cuda:0") for p, _ in sweeps]
    torch.cuda.synchronize()
    work = (corner, surf, sweeps, d_sweeps)
    info = card_info()

    # (c), (d): the library's begin_sweep trace on stderr, captured from the file descriptor
    log = tempfile.NamedTemporaryFile(prefix="map_update_trace_", suffix=".log", delete=False)
    saved = os.dup(2)
    sys.stderr.flush()
    os.dup2(log.fileno(), 2)
    busy = []
    try:
        for _ in range(args.windows):
            print("@@window", file=sys.stderr, flush=True)
            _, ss = run_window(api, work, args.warmup, args.steps)
            busy.append([round(1e3 * float(v) / args.steps, 4) for v in ss["busy"]])
    finally:
        sys.stderr.flush()
        os.dup2(saved, 2)
        os.close(saved)
    text = open(log.name).read()
    os.unlink(log.name)
    waits, sizes = [], []
    for chunk in text.split("@@window")[1:]:
        lines = [m for m in (BEGIN_RE.search(ln) for ln in chunk.splitlines()) if m]
        for m in lines[args.warmup:]:
            waits.append(float(m.group(1)))
            sizes.append([int(m.group(i)) for i in (2, 3, 4, 5)])
    s_corner = [a + c for a, _, c, _ in sizes]
    s_surf = [b + d for _, b, _, d in sizes]

    # (a), (b): one more window under the profiler
    from torch.profiler import ProfilerActivity, profile
    prof = profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA])
    run_window(api, work, args.warmup, args.steps, profiler=prof)
    trace = os.path.join(args.out, "timeline.pt.trace.json")
    prof.export_chrome_trace(trace)
    rows, n_streams = analyse_trace(trace)

    summary = {
        "card": info, "workload": "hdl64_1m", "warmup": args.warmup, "steps": args.steps, "windows": args.windows,
        "update_chain": "multi-launch" if args.split_update else "default",
        "a_update": {"sweeps_seen": len(rows), "update_streams": n_streams,
                     "span_us_median": med([r["span_us"] for r in rows]),
                     "span_us_min_max": [min(r["span_us"] for r in rows), max(r["span_us"] for r in rows)] if rows else None,
                     "longest_stream_span_us_median": med([r["stream_spans_us"][0] for r in rows]),
                     "ops_median": med([r["ops"] for r in rows]), "kernels_median": med([r["kernels"] for r in rows]),
                     "kernel_us_median": med([r["kernel_us"] for r in rows])},
        "b_launch_latency_us_median": med([r["launch_latency_us"] for r in rows if r["launch_latency_us"] is not None]),
        "c_begin_sweep_wait_us": {"median": med(waits), "min_max": [min(waits), max(waits)] if waits else None,
                                  "n": len(waits)},
        "d_sizes": {"n_ins_corner_surf_median": [med([s[0] for s in sizes]), med([s[1] for s in sizes])],
                    "n_raw_corner_surf_median": [med([s[2] for s in sizes]), med([s[3] for s in sizes])],
                    "n_raw_corner_surf_max": [max(s[2] for s in sizes), max(s[3] for s in sizes)] if sizes else None,
                    "S_max_corner_surf": [max(s_corner), max(s_surf)] if sizes else None,
                    "sweeps_with_S_over_CS_MAX_N": sum(1 for a, b in zip(s_corner, s_surf) if max(a, b) > CS_MAX_N),
                    "sweeps": len(sizes)},
        "streaming_busy_ms_per_sweep_reg_odom_map": busy,
        "per_sweep": rows,
    }
    with open(os.path.join(args.out, "summary.json"), "w") as f:
        json.dump(summary, f, indent=1)
    short = {k: v for k, v in summary.items() if k != "per_sweep"}
    short["per_sweep_example"] = rows[len(rows) // 2] if rows else None
    print(json.dumps(short, indent=1))


if __name__ == "__main__":
    main()
