"""Headless CLI of the export path (the reference drives it from a wx menu, master/DesignCSG.cpp:812-1031).

    python -m designcsg_b200 compile DESIGN.py SCENE_DIR              design script -> scene files ("Run")
    python -m designcsg_b200 export  SCENE_DIR|DESIGN.py [--level L] [--ply P] [--stl S] [--normals]
    python -m designcsg_b200 export  SCENE_DIR|DESIGN.py --ply-indexed P [--normals] [--level L]
                                                                       indexed binary PLY (shared float vertices, optional
                                                                       normals; not the reference's format)
    ... export ... --outward                                           every triangle wound to face out of the solid (any of
                                                                       the files above; not the reference's bytes)
    python -m designcsg_b200 inspect SCENE_DIR|DESIGN.py [--level L] [--outward] [--components]
                                                                       one JSON line: edge topology, shells, area, volume,
                                                                       centroid and extents of the mesh --ply-indexed writes
    ... inspect ... --deviation [--subdivision K] [--tolerance T]     ... and the design's SDF sampled over that mesh
    torchrun --nproc-per-node G -m designcsg_b200 export ...          z-slab sharded over G GPUs (dcsg_export_sharded; the
                                                                       same export from a C host: tools/dcsg_mgpu.c)
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np


def _scene_dir(path):
    from . import api
    if os.path.isdir(path):
        return path
    out = tempfile.mkdtemp(prefix="dcsg_scene_")
    return api.compile_design(path, out)


def cmd_compile(args):
    from . import api
    print(api.compile_design(args.design, args.scene_dir))


def _export_config(scene):
    """exportConfig.txt as the reference parses it (DesignCSG.cpp:827-835); a design that never called setExportConfig has
    none -- then the CLI needs --level (the reference's GUI refuses to export such a design, too)."""
    path = os.path.join(scene, "exportConfig.txt")
    if not os.path.exists(path):
        return None
    cfg = open(path).read().split("\n")
    if len(cfg) < 6:
        raise SystemExit("%s: expected at least 6 lines (setExportConfig writes 9)" % path)
    return cfg


def _export_levels(scene, level_override):
    """(exportConfig.txt lines or None, search diameter, projection steps, minimum / maximum octree level, grid level,
    complex-surface threshold) of an export; level_override L > 0 = uniform lattice of 2^L cells per side."""
    cfg = _export_config(scene)
    if cfg is None and not level_override:
        raise SystemExit("%s has no exportConfig.txt (the design never called setExportConfig): pass --level L" % scene)
    # exportConfig.txt lines 1-6: search diameter, minimum / maximum octree level, grid level, complex-surface threshold,
    # projection steps
    search, steps = (float(cfg[0]), int(cfg[5])) if cfg else (10.0, 50)
    lo, hi, level, threshold = (int(cfg[1]), int(cfg[2]), int(cfg[3]), float(cfg[4])) if cfg else (0, 0, 0, float(np.pi / 4))
    if level_override:
        lo = hi = level = level_override
    return cfg, search, steps, lo, hi, level, threshold


def cmd_export(args):
    from . import api, build
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.ply_indexed:
        # checked before anything is built or a device is touched
        if args.ply or args.stl:
            raise SystemExit("--ply-indexed cannot be combined with --ply / --stl: the two exports would project the mesh twice, "
                             "and the indexed file welds an adaptive mesh before its projection; run them separately")
        if args.no_retopologize:
            raise SystemExit("--ply-indexed re-encodes the reference's export, which always retopologizes: drop --no-retopologize")
        if world > 1 and not args.level:
            raise SystemExit("--ply-indexed on several GPUs needs --level L (a uniform lattice): the weld of an adaptive mesh "
                             "spans the GPUs' slabs")
    build.build()                       # serialised across the ranks of a node by a file lock; the first one compiles
    scene = _scene_dir(args.scene)
    cfg, search, steps, lo, hi, level, threshold = _export_levels(scene, args.level)
    t0 = time.perf_counter()
    ctx = api.Context(local)
    ctx.build(scene)
    t_build = time.perf_counter() - t0
    report = {"scene": scene, "octree_levels": [lo, hi, level], "gd_steps": steps, "gpus": world, "build_s": t_build}
    if world == 1 and args.ply_indexed:
        t1 = time.perf_counter()
        rep = ctx.export_indexed(scene, args.level, args.ply_indexed, normals=args.normals, outward=args.outward)
        report.update(triangles=int(rep.num_triangles), vertices=int(rep.num_vertices), box=[float(v) for v in rep.box],
                      export_s=time.perf_counter() - t1, project_and_write_ms=float(rep.write_ms))
    elif world == 1:
        box = ctx.bbox(search)
        report["box"] = [float(v) for v in box]
        pipelined = not args.normals                       # projection pipelined with formatting, D2H and the file writes
        mesh = ctx.extract(box, level, gd_steps=steps, want_normals=args.normals, copy_to_host=False, min_level=lo, max_level=hi,
                           complex_threshold=threshold, retopologize=not args.no_retopologize, defer_projection=pipelined)
        report.update(triangles=mesh.num_triangles, vertices=mesh.num_vertices, stage_ms=mesh.stage_ms)
        t1 = time.perf_counter()
        if args.outward:
            mesh.orient()
        if pipelined:
            mesh.project_and_write_files(steps, args.stl, args.ply)
        else:
            if args.ply:
                mesh.write_ply(args.ply)
            if args.stl:
                mesh.write_stl(args.stl)
        report["project_and_write_s" if pipelined else "write_s"] = time.perf_counter() - t1
        mesh.free()
    else:
        import torch
        import torch.distributed as dist
        from . import distributed as D
        if args.normals and not args.ply_indexed:
            raise SystemExit("--normals has no effect on the files (the reference's writers store no normals) and is not "
                             "supported by the sharded export; drop it or run on one GPU")
        if not cfg:
            raise SystemExit("the sharded export reads exportConfig.txt; this design has none")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        comm = D.create_comm(ctx)       # from here on everything collective happens inside libdcsg
        t1 = time.perf_counter()
        if args.ply_indexed:
            rep = comm.export_indexed(scene, args.level, args.ply_indexed, normals=args.normals, outward=args.outward)
        else:
            rep = comm.export(scene, args.level, args.stl, args.ply, outward=args.outward)
        report.update(triangles=int(rep.num_triangles), vertices=int(rep.num_vertices), box=[float(v) for v in rep.box],
                      export_s=time.perf_counter() - t1, search_ms=float(rep.bbox_ms), project_and_write_ms=float(rep.write_ms))
        comm.close()
        dist.destroy_process_group()
    ctx.close()
    report["total_s"] = time.perf_counter() - t0
    if rank == 0:
        print(json.dumps(report))


def cmd_inspect(args):
    """The report of dcsg_mesh_inspect on the mesh `export --ply-indexed` writes with the same options: extraction (the
    export's levels, threshold and retopologize), --outward orientation, the weld of adaptive levels, the projection."""
    from . import api, build
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        raise SystemExit("inspect runs on one GPU: the mesh of a sharded export is never gathered; run it without torchrun")
    if not 1 <= args.subdivision <= 16:
        raise SystemExit("--subdivision must be in 1..16, not %d" % args.subdivision)
    if args.tolerance is not None and not args.tolerance >= 0.0:
        raise SystemExit("--tolerance must be a number >= 0, not %r" % args.tolerance)
    build.build()
    scene = _scene_dir(args.scene)
    _, search, steps, lo, hi, level, threshold = _export_levels(scene, args.level)
    ctx = api.Context(int(os.environ.get("LOCAL_RANK", "0")))
    ctx.build(scene)
    box = ctx.bbox(search)
    mesh = ctx.extract(box, level, copy_to_host=False, min_level=lo, max_level=hi, complex_threshold=threshold,
                       retopologize=True, defer_projection=True)
    if args.outward:
        mesh.orient()
    if not (lo >= level and hi == level):
        mesh.weld()
    ctx.project(mesh, steps)
    report = mesh.inspect(components=args.components)
    for name in ("component_triangles", "component_area", "component_signed_volume"):
        if name in report:
            report[name] = report[name].tolist()
    report.update(scene=scene, octree_levels=[lo, hi, level], gd_steps=steps, outward=bool(args.outward))
    if args.deviation:
        cell = float(max(box[3:6])) / (1 << level)          # the finest lattice cell
        tolerance = cell / 10 if args.tolerance is None else args.tolerance
        dev = mesh.deviation(args.subdivision, tolerance)
        dev.update(subdivision=args.subdivision, tolerance=tolerance, cell=cell)
        report["deviation"] = dev
    mesh.free()
    ctx.close()
    print(json.dumps(report))


def main():
    ap = argparse.ArgumentParser(prog="python -m designcsg_b200")
    sub = ap.add_subparsers(dest="cmd", required=True)
    c = sub.add_parser("compile")
    c.add_argument("design")
    c.add_argument("scene_dir")
    c.set_defaults(fn=cmd_compile)
    e = sub.add_parser("export")
    e.add_argument("scene", help="scene directory or design script")
    e.add_argument("--level", type=int, default=0, help="uniform lattice of 2^L cells per side (default: the octree levels of "
                   "exportConfig.txt, adaptive walk + retopologize like the reference's Export)")
    e.add_argument("--no-retopologize", action="store_true", help="skip cms::retopologize (identity for uniform lattices)")
    e.add_argument("--ply")
    e.add_argument("--stl")
    e.add_argument("--ply-indexed", help="write an indexed binary PLY instead (shared float vertices; with --normals the "
                   "projection's normals too) -- a format beyond the reference's")
    e.add_argument("--normals", action="store_true")
    e.add_argument("--outward", action="store_true", help="wind every triangle to face out of the solid (dcsg_mesh_orient) in "
                   "whichever files are written; the files are then not the reference's bytes, whose winding is mixed")
    e.set_defaults(fn=cmd_export)
    i = sub.add_parser("inspect", help="report on the mesh `export --ply-indexed` would write (one JSON line)")
    i.add_argument("scene", help="scene directory or design script")
    i.add_argument("--level", type=int, default=0, help="uniform lattice of 2^L cells per side (default: exportConfig.txt's levels)")
    i.add_argument("--outward", action="store_true", help="orient the mesh first, as export --outward does")
    i.add_argument("--components", action="store_true", help="add per-shell triangle counts, areas and signed volumes")
    i.add_argument("--deviation", action="store_true", help="add the design's SDF sampled over every triangle (dcsg_mesh_deviation)")
    i.add_argument("--subdivision", type=int, default=4, help="--deviation: samples at (i, j) / K over each triangle, K in 1..16 "
                   "(default 4)")
    i.add_argument("--tolerance", type=float, default=None, help="--deviation: |SDF| above which a triangle counts as over "
                   "tolerance (default: a tenth of the finest lattice cell)")
    i.set_defaults(fn=cmd_inspect)
    args = ap.parse_args()
    args.fn(args)


if __name__ == "__main__":
    main()
