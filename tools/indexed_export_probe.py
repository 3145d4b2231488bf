"""Wall time and file size of the indexed PLY against the reference's soup files, on one GPU.

    python tools/indexed_export_probe.py [--runs 5] [--out profiles/indexed_export.jsonl]

Workloads: Design1 at 1024^3 (uniform lattice), Design1 and Design2 at their shipped octree levels (adaptive walk +
retopologize).  Per workload the four arms -- dcsg_export writing the PLY alone, dcsg_export writing PLY + STL,
dcsg_export_indexed without and with normals -- are alternated, each run into fresh files in a temporary directory that are
removed right after (so every run writes new pages, as a user's export does).  Every export call compiles the scene with
NVRTC first (dcsg_build), which takes longer than the rest, so two numbers are kept: write_ms = the report's time from the
extracted mesh to complete files (the soup arms: projection + formatting + copies + writes; the indexed arms: weld + the same),
and call_ms = host clock around the whole synchronous call (build, search, extraction, files).
The weld is timed on its own through the stepwise API (extract with defer_projection, then Mesh.weld(), which ends in a
device synchronise).  One JSON line per workload and arm, plus one per workload for the weld, each with the GPU's name,
power limit and max SM clock read in the same run."""
import argparse
import json
import os
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


def run_arm(ctx, scene, level, arm, tmp):
    ply, stl = os.path.join(tmp, "o.ply"), os.path.join(tmp, "o.stl")
    t0 = time.perf_counter()
    if arm == "soup_ply":
        rep = ctx.export(scene, level, ply_path=ply)
    elif arm == "soup_ply_stl":
        rep = ctx.export(scene, level, stl_path=stl, ply_path=ply)
    else:
        rep = ctx.export_indexed(scene, level, ply, normals=arm == "indexed_normals")
    ms = (time.perf_counter() - t0) * 1e3
    size = sum(os.path.getsize(p) for p in (ply, stl) if os.path.exists(p))
    for p in (ply, stl):
        if os.path.exists(p):
            os.remove(p)
    return ms, size, rep


def weld_probe(ctx, name, level, runs):
    cfg = scenes.materialize(name)["export_config"]
    search, lo, hi, grid, thr = float(cfg[0]), int(cfg[1]), int(cfg[2]), int(cfg[3]), float(cfg[4])
    if level:
        lo = hi = grid = level
    box = ctx.bbox(search)
    times, before, after = [], 0, 0
    mesh = None
    for _ in range(runs + 1):
        mesh = ctx.extract(box, grid, min_level=lo, max_level=hi, complex_threshold=thr, retopologize=True, defer_projection=True,
                           copy_to_host=False, mesh=mesh)
        before = mesh.num_vertices
        t0 = time.perf_counter()
        mesh.weld()
        times.append((time.perf_counter() - t0) * 1e3)
        after = mesh.num_vertices
    triangles = mesh.num_triangles
    mesh.free()
    return {"weld_ms_median": statistics.median(times[1:]), "weld_ms_runs": times[1:], "vertices_before_weld": before,
            "vertices_after_weld": after, "triangles": triangles}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out", default=os.path.join("profiles", "indexed_export.jsonl"))
    args = ap.parse_args()
    build.build()
    hw = gpu_info()
    arms = ("soup_ply", "soup_ply_stl", "indexed", "indexed_normals")
    lines = []
    for name, level in WORKLOADS:
        scene = scenes.materialize(name)["dir"]
        ctx = api.Context(0)
        ctx.build(scene)
        label = "%s %s" % (name, "%d^3 uniform" % (1 << level) if level else "shipped levels")
        weld = weld_probe(ctx, name, level, args.runs)
        lines.append(dict(hw, workload=label, arm="weld", **weld))
        print(json.dumps(lines[-1]), flush=True)
        times = {a: [] for a in arms}
        calls = {a: [] for a in arms}
        info = {}
        with tempfile.TemporaryDirectory(prefix="dcsg_probe_") as tmp:
            for a in arms:                                  # warm-up: module loads, buffer growth, page cache state
                run_arm(ctx, scene, level, a, tmp)
            for _ in range(args.runs):
                for a in arms:
                    ms, size, rep = run_arm(ctx, scene, level, a, tmp)
                    times[a].append(float(rep.write_ms))
                    calls[a].append(ms)
                    info[a] = {"file_bytes": size, "vertices": int(rep.num_vertices), "triangles": int(rep.num_triangles)}
        for a in arms:
            lines.append(dict(hw, workload=label, arm=a, write_ms_median=statistics.median(times[a]), write_ms_runs=times[a],
                              call_ms_median=statistics.median(calls[a]), **info[a]))
            print(json.dumps(lines[-1]), flush=True)
        ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
