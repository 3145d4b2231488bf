"""Cost of the mesh deviation (dcsg_mesh_deviation) on one GPU, and what it finds on the shipped designs.

    python tools/deviation_probe.py [--runs 7] [--out profiles/deviation.jsonl]

dcsg_mesh_deviation timed with CUDA events around the whole synchronous call on the library's stream (a torch stream handed
over with dcsg_set_stream), median of `runs` calls after one warm-up call that grows the buffers, at subdivisions k = 1, 4 and
8: Design1 at 1024^3 (uniform lattice, oriented, 50 projection steps) and Design1 / Design2 at their shipped octree levels
(adaptive walk + retopologize, oriented, welded, projected) -- the meshes `inspect --outward` measures.  The rate is SDF
evaluations (every vertex plus S = (k+1)(k+2)/2 - 3 points per triangle) per second, set against the lattice pass's rate on
the same design at 1024^3 (dcsg_mesh.lattice_samples over its stage time, on a second extraction after a warm-up one).  The
reports go with the timings.  One JSON line per measurement, each with the GPU's name, power limit and max SM clock read in
the same run."""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from designcsg_b200 import api, build       # noqa: E402
from tests.golden import scenes              # noqa: E402
from tools.inspect_probe import exported_mesh, gpu_info, levels      # noqa: E402

WORKLOADS = [("design1", 10), ("design1", 0), ("design2", 0)]      # level 0 = the design's exportConfig.txt
SUBDIVISIONS = (1, 4, 8)


def deviation_probe(torch, stream, mesh, k, tolerance, runs):
    events = []
    report = None
    for _ in range(runs + 1):                       # the first run grows the buffers
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream.synchronize()
        a.record(stream)
        report = mesh.deviation(k, tolerance)
        b.record(stream)
        b.synchronize()
        events.append(a.elapsed_time(b))
    return {"deviation_ms_median": statistics.median(events[1:]), "deviation_ms_runs": events[1:], "report": report}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--out", default=os.path.join("profiles", "deviation.jsonl"))
    args = ap.parse_args()
    import torch
    build.build()
    hw = gpu_info()
    lines = []

    def emit(line):
        lines.append(dict(hw, **line))
        print(json.dumps(lines[-1]), flush=True)

    for name in sorted({n for n, _ in WORKLOADS}):
        ctx = api.Context(0)
        ctx.build(scenes.materialize(name)["dir"])
        stream = torch.cuda.Stream()
        ctx.set_stream(stream.cuda_stream)
        box = ctx.bbox(10.0)
        ctx.extract(box, 10, copy_to_host=False).free()      # warm-up: module load, buffers
        lattice = ctx.extract(box, 10, copy_to_host=False)
        stream.synchronize()
        lattice_rate = lattice.c.lattice_samples / (lattice.stage_ms["lattice"] * 1e-3)
        emit(dict(workload="%s 1024^3 lattice pass" % name, arm="lattice", evaluations=int(lattice.c.lattice_samples),
                  lattice_ms=lattice.stage_ms["lattice"], evals_per_s=lattice_rate))
        lattice.free()
        for wname, level in WORKLOADS:
            if wname != name:
                continue
            mesh = exported_mesh(ctx, name, level)
            search, lo, hi, grid, thr, steps = levels(name, level)
            box = ctx.bbox(search)
            cell = float(max(box[3:6])) / (1 << grid)
            label = "%s %s" % (name, "%d^3 uniform" % (1 << level) if level else "shipped levels, welded")
            for k in SUBDIVISIONS:
                evals = mesh.num_vertices + mesh.num_triangles * ((k + 1) * (k + 2) // 2 - 3)
                r = deviation_probe(torch, stream, mesh, k, cell / 10, args.runs)
                emit(dict(workload=label, arm="dcsg_mesh_deviation", k=k, tolerance=cell / 10, cell=cell, triangles=mesh.num_triangles,
                          vertices=mesh.num_vertices, evaluations=evals, evals_per_s=evals / (r["deviation_ms_median"] * 1e-3),
                          lattice_evals_per_s=lattice_rate, **r))
            mesh.free()
        ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
