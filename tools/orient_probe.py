"""Cost of the outward winding (dcsg_mesh_orient) on one GPU.

    python tools/orient_probe.py [--runs 7] [--out profiles/orient.jsonl]

1. dcsg_mesh_orient alone, timed with CUDA events on the library's stream (a torch stream handed over with dcsg_set_stream):
   Design1 at 1024^3 (uniform lattice) and Design1 / Design2 at their shipped octree levels (adaptive walk + retopologize).  A
   second call on an oriented mesh does nothing, so every run orients a fresh extraction into the same mesh object; the
   triangles were just written by that extraction, as in an export.  The window holds the two kernels, cub's scan and the
   4-byte read-back of the check; call_ms is the host clock around the whole (synchronous) call.
2. The bench's export_to_files step on Design1 at 1024^3 -- search, extraction (projection deferred), then projection pipelined
   with formatting, copies and the writes of the PLY and STL into a temporary directory -- without and with Mesh.orient()
   between the extraction and the file pipeline, the two arms alternated in one process.
One JSON line per measurement, each with the GPU's name, power limit and max SM clock read in the same run."""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from designcsg_b200 import api, build       # noqa: E402
from tests.golden import scenes              # noqa: E402

WORKLOADS = [("design1", 10), ("design1", 0), ("design2", 0)]      # level 0 = the design's exportConfig.txt


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         stdout=subprocess.PIPE, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def levels(name, level):
    cfg = scenes.materialize(name)["export_config"]
    search, lo, hi, grid, thr, steps = float(cfg[0]), int(cfg[1]), int(cfg[2]), int(cfg[3]), float(cfg[4]), int(cfg[5])
    if level:
        lo = hi = grid = level
    return search, lo, hi, grid, thr, steps


def orient_probe(torch, ctx, stream, name, level, runs):
    search, lo, hi, grid, thr, _ = levels(name, level)
    box = ctx.bbox(search)
    mesh = None
    events, calls = [], []
    for _ in range(runs + 1):                       # the first run grows the buffers
        mesh = ctx.extract(box, grid, min_level=lo, max_level=hi, complex_threshold=thr, retopologize=True, defer_projection=True,
                           copy_to_host=False, mesh=mesh)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream.synchronize()
        a.record(stream)
        t0 = time.perf_counter()
        mesh.orient()
        calls.append((time.perf_counter() - t0) * 1e3)
        b.record(stream)
        b.synchronize()
        events.append(a.elapsed_time(b))
    out = {"orient_ms_median": statistics.median(events[1:]), "orient_ms_runs": events[1:],
           "call_ms_median": statistics.median(calls[1:]), "cells": mesh.num_cells, "triangles": mesh.num_triangles}
    mesh.free()
    return out


def export_to_files(ctx, mesh, level, steps, outward, out_dir):
    ply, stl = os.path.join(out_dir, "o.ply"), os.path.join(out_dir, "o.stl")
    t0 = time.perf_counter()
    box = ctx.bbox(10.0)
    ctx.extract(box, level, gd_steps=steps, copy_to_host=False, mesh=mesh, defer_projection=True)
    if outward:
        mesh.orient()
    mesh.project_and_write_files(steps, stl, ply)
    ms = (time.perf_counter() - t0) * 1e3
    for p in (ply, stl):
        os.remove(p)
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--out", default=os.path.join("profiles", "orient.jsonl"))
    args = ap.parse_args()
    import torch
    build.build()
    hw = gpu_info()
    lines = []
    for name, level in WORKLOADS:
        ctx = api.Context(0)
        ctx.build(scenes.materialize(name)["dir"])
        stream = torch.cuda.Stream()
        ctx.set_stream(stream.cuda_stream)
        label = "%s %s" % (name, "%d^3 uniform" % (1 << level) if level else "shipped levels")
        lines.append(dict(hw, workload=label, arm="dcsg_mesh_orient", **orient_probe(torch, ctx, stream, name, level, args.runs)))
        print(json.dumps(lines[-1]), flush=True)
        if name == "design1" and level:
            mesh = api.Mesh(ctx)
            times = {False: [], True: []}
            out_dir = tempfile.mkdtemp(prefix="dcsg_orient_probe_")
            try:
                for outward in (False, True):               # warm-up
                    export_to_files(ctx, mesh, level, 50, outward, out_dir)
                for _ in range(args.runs):
                    for outward in (False, True):
                        times[outward].append(export_to_files(ctx, mesh, level, 50, outward, out_dir))
            finally:
                shutil.rmtree(out_dir, ignore_errors=True)
            triangles = mesh.num_triangles
            mesh.free()
            for outward in (False, True):
                lines.append(dict(hw, workload=label, arm="export_to_files" + ("_outward" if outward else ""),
                                  ms_median=statistics.median(times[outward]), ms_runs=times[outward], triangles=triangles))
                print(json.dumps(lines[-1]), flush=True)
        ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
