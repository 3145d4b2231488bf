"""Cost of the mesh report (dcsg_mesh_inspect) on one GPU, and what it finds on the shipped designs.

    python tools/inspect_probe.py [--runs 7] [--out profiles/inspect.jsonl]

1. dcsg_mesh_inspect alone, timed with CUDA events on the library's stream (a torch stream handed over with dcsg_set_stream)
   and with the host clock around the whole synchronous call, after one warm-up call that grows the buffers: Design1 at
   1024^3 (uniform lattice, oriented, 50 projection steps) and Design1 / Design2 at their shipped octree levels (adaptive walk
   + retopologize, oriented, welded, projected) -- the meshes `export --ply-indexed --outward` writes.  The call is pure, so
   every run inspects the same mesh; its arrays (and most of the scratch) fit in L2 only for the shipped levels.
2. The reports themselves: the timed meshes, and Design1 / Design2 / stress at 128^3 with and without the centre-sample cull.
One JSON line per measurement, each with the GPU's name, power limit and max SM clock read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from designcsg_b200 import api, build       # noqa: E402
from tests.golden import scenes              # noqa: E402

WORKLOADS = [("design1", 10), ("design1", 0), ("design2", 0)]      # level 0 = the design's exportConfig.txt
FINDINGS = [("design1", 7), ("design2", 7), ("stress", 7)]


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         stdout=subprocess.PIPE, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def levels(name, level):
    cfg = scenes.materialize(name)["export_config"]
    search, lo, hi, grid, thr, steps = float(cfg[0]), int(cfg[1]), int(cfg[2]), int(cfg[3]), float(cfg[4]), int(cfg[5])
    if level:
        lo, hi, grid, steps = level, level, level, 50
    return search, lo, hi, grid, thr, steps


def exported_mesh(ctx, name, level):
    """The mesh `export --ply-indexed --outward` writes."""
    search, lo, hi, grid, thr, steps = levels(name, level)
    mesh = ctx.extract(ctx.bbox(search), grid, min_level=lo, max_level=hi, complex_threshold=thr, retopologize=True,
                       defer_projection=True, copy_to_host=False)
    mesh.orient()
    if not level:
        mesh.weld()
    ctx.project(mesh, steps)
    return mesh


def inspect_probe(torch, ctx, stream, mesh, runs):
    events, calls = [], []
    report = None
    for _ in range(runs + 1):                       # the first run grows the buffers
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream.synchronize()
        a.record(stream)
        t0 = time.perf_counter()
        report = mesh.inspect()
        calls.append((time.perf_counter() - t0) * 1e3)
        b.record(stream)
        b.synchronize()
        events.append(a.elapsed_time(b))
    return {"inspect_ms_median": statistics.median(events[1:]), "inspect_ms_runs": events[1:],
            "call_ms_median": statistics.median(calls[1:]), "report": report}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--out", default=os.path.join("profiles", "inspect.jsonl"))
    args = ap.parse_args()
    import torch
    build.build()
    hw = gpu_info()
    lines = []

    def emit(line):
        lines.append(dict(hw, **line))
        print(json.dumps(lines[-1]), flush=True)

    contexts = {}
    for name in sorted({n for n, _ in WORKLOADS + FINDINGS}):
        ctx = api.Context(0)
        ctx.build(scenes.materialize(name)["dir"])
        stream = torch.cuda.Stream()
        ctx.set_stream(stream.cuda_stream)
        contexts[name] = (ctx, stream)
    for name, level in WORKLOADS:
        ctx, stream = contexts[name]
        mesh = exported_mesh(ctx, name, level)
        label = "%s %s" % (name, "%d^3 uniform" % (1 << level) if level else "shipped levels, welded")
        emit(dict(workload=label, arm="dcsg_mesh_inspect", triangles=mesh.num_triangles, vertices=mesh.num_vertices,
                  **inspect_probe(torch, ctx, stream, mesh, args.runs)))
        mesh.free()
    for name, level in FINDINGS:
        ctx, _ = contexts[name]
        for no_cull in (False, True):
            mesh = ctx.extract(ctx.bbox(10.0), level, gd_steps=50, no_cull=no_cull, copy_to_host=False)
            mesh.orient()
            emit(dict(workload="%s %d^3 uniform, oriented, cull %s" % (name, 1 << level, "off" if no_cull else "on"), arm="report",
                      report=mesh.inspect()))
            mesh.free()
    for ctx, _ in contexts.values():
        ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
