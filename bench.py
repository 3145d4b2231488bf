#!/usr/bin/env python
"""bench.py -- the contract benchmark of the DesignCSG export hot path on B200.

    python bench.py --gpus 1 --steps K --warmup W                      (our arm, one GPU)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W                      (our arm, z-slabs over N GPUs)
    python bench.py --impl reference --gpus N --steps K --warmup W     (the reference's CPU path, host cores)
    python bench.py ... --dump-outputs DIR                             (also write the last timed step's results as .npy)

Metric (BASELINE.json): SDF voxels/s of a whole export at 1024^3.  Workload: Design1 (the reference's shipped
design, replayed from tests/golden/design1/capture.json through our front-end) on the 1024^3 cell lattice,
uniform octree levels 10/10/10, 50 gradient-descent steps -- BASELINE config 4; it fits one GPU, so the same
workload is used for every N (strong scaling).  One step = one pass of the hot path: 256^3 bounding-box search
-> lattice evaluation (octree-ordered: the samples the reference's walk touches) -> classify / compact ->
vertex + triangle emission -> 50-step projection
(N > 1, through libdcsg's communicator: sharded search with its all-reduce, all-gather of the slabs' counts, the
projected mesh stored by the kernels into rank 0's arrays over NVLink -- the whole mesh is complete on rank 0 when
the step ends).

  value  voxels/s with the compiled scene resident on the device and the mesh left in HBM
  e2e    the same pass through the C ABI with HOST buffers: side table uploaded every step, every rank's byte
         ranges of the byte-exact PLY + STL files in pinned host memory every step (wall clock, max over ranks)
  roofline / roofline_other     the two SDF stages (projection; octree-ordered lattice evaluation) against the
                                measured non-tensor FP32 rate; roofline_dense_lattice = the dense lattice kernel
  cpu_baseline                  the reference's own code (oracle/_ref) on a bounded sample, host cores
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

FLOP_PER_EVAL = {"design1": 287.0, "design2": 1090.0}      # SURVEY.md 8(d); DESIGN.md "Rooflines"
FLOP_PER_NORMAL_EXTRA = 22.0                               # differences, scale, normalize, position update
# floating-point operations the checked fast copy actually EXECUTES per evaluation (same counting rule, from the SASS of the
# projection's tap loop: 39 FMUL + 33 FADD + 18 FFMA x 2 + 30 FSETP + 9 MUFU + ~7 FP64 / min-max): the zero terms of the
# axis-aligned transforms are not executed at all (DESIGN.md 3b), so `achieved` (the reference's operations per second) is
# larger than the rate the FP pipes really run at
EXECUTED_FLOP_PER_EVAL = {"design1": 154.0}
SEARCH_DIAMETER = 10.0                                     # exportConfig.txt line 1 of every shipped design


# ---------------------------------------------------------------------------------------------------------------
# clocks during the timed region (recipe of B200_PROFILING.md)
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc, self.thread = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 6:
                self.samples.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# the reference's CPU path on a bounded sample of the workload
# ---------------------------------------------------------------------------------------------------------------
def use_all_host_threads():
    """The reference's evaluator stand-in is an OpenMP loop (oracle/ref_driver.cpp); torch.distributed.run exports
    OMP_NUM_THREADS=1 to every rank, which would time the reference single-threaded at N > 1.  Set it explicitly, before
    the oracle library (and with it libgomp) is loaded, to all host cores -- the same at every N -- and report it."""
    n = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(n)
    return n


class CpuReferenceSample:
    """The reference's export on a FIXED, stratified sample of 128^3-cell blocks of the 2^level lattice.

    A block is an octree node of level (level-7) of the export's own octree; meshing it with grid level 7 visits exactly
    the cells, lattice samples and triangles the full export visits inside that block (cms::Mesh::getSurface,
    cms::performGradientDescent through oracle/_ref when built from the reference's sources, else the C++ port).
    Blocks differ in cost by orders of magnitude (the walk leaves an empty block after one sample), so the sample is
    stratified: every block is classified once, untimed, by the reference's own walk at 16^3 cells per block, and
    `blocks` of them are picked from the surface and the empty stratum in their true proportion -- evenly spaced, the
    surface blocks in the order of their coarse triangle count, i.e. at the quantiles of the cost distribution.  The
    choice depends on the scene only: every step of every run times the same blocks.  The 256^3 bounding-box search is
    timed once and charged pro rata."""

    def __init__(self, scene_name, level, gd_steps, blocks):
        self.threads = use_all_host_threads()
        from oracle.oracle import Oracle
        from oracle import build as obuild
        from tests.golden import scenes
        scene = scenes.materialize(scene_name)
        self.kind = "reference" if (obuild.have_reference() or os.path.exists(obuild.ref_lib_path(scene_name))) else "port"
        self.orc = Oracle.for_scene(scene, self.kind)
        self.level, self.gd_steps = level, gd_steps
        t0 = time.perf_counter()
        self.box = self.orc.bbox(SEARCH_DIAMETER)
        self.t_bbox = time.perf_counter() - t0
        self.per_side = 1 << (level - 7)
        total = self.per_side ** 3
        coarse = [len(self.orc.get_surface(self.block_box(p), 4, 4, 4)) for p in range(total)]
        # surface blocks ordered by how much surface they hold, so that evenly spaced picks are quantiles of the cost
        surface = sorted((p for p in range(total) if coarse[p]), key=lambda p: (coarse[p], p))
        empty = [p for p in range(total) if not coarse[p]]
        blocks = min(blocks, total)
        n_surface = min(len(surface), max(1 if surface else 0, int(round(blocks * len(surface) / total))))
        n_empty = min(len(empty), blocks - n_surface)
        spaced = lambda items, k: [items[int((i + 0.5) * len(items) / k)] for i in range(k)]
        self.picks = sorted(spaced(surface, n_surface) + spaced(empty, n_empty))
        self.strata = (len(surface), total, n_surface, n_empty)

    def block_box(self, p):
        ps, box = self.per_side, self.box
        side = box[3] / ps
        bz, by, bx = p // (ps * ps), (p // ps) % ps, p % ps
        centre = box[:3] - box[3] / 2 + (np.array([bx, by, bz], dtype=np.float64) + 0.5) * side
        return np.array([centre[0], centre[1], centre[2], side, side, side], dtype=np.float32)

    def run(self):
        """One pass over the sample; returns (seconds incl. the pro-rata search, voxels, triangles)."""
        tris = 0
        t0 = time.perf_counter()
        for p in self.picks:
            soup = self.orc.get_surface(self.block_box(p), 7, 7, 7)
            if len(soup):
                self.orc.gradient_descent(soup, self.gd_steps)
            tris += len(soup)
        seconds = time.perf_counter() - t0 + self.t_bbox * len(self.picks) / self.per_side ** 3
        return seconds, len(self.picks) * 128 ** 3, tris

    def describe(self, seconds, voxels, tris, passes=1):
        s, total, ns, ne = self.strata
        return {"value": voxels / seconds, "unit": "voxels/s", "cores": os.cpu_count(), "threads": self.threads, "kind": self.kind,
                "sample": "fixed stratified sample of the %d^3 lattice: %d surface + %d empty 128^3-cell blocks (%d of %d blocks "
                          "hold surface; blocks %s), %d triangles per pass, %d pass(es) in %.1f s; bbox search %.2f s charged pro "
                          "rata; OMP_NUM_THREADS=%d" % (1 << self.level, ns, ne, s, total, self.picks, tris, passes, seconds,
                                                        self.t_bbox, self.threads),
                "seconds": seconds}


def cpu_reference_sample(scene_name, level, gd_steps, blocks):
    sample = CpuReferenceSample(scene_name, level, gd_steps, blocks)
    seconds, voxels, tris = sample.run()
    return sample.describe(seconds, voxels, tris)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = CpuReferenceSample(args.scene, args.level, args.gd_steps, args.cpu_blocks)
    timed = []
    for i in range(args.warmup + args.steps):
        last = sample.run()                                   # every step times the same blocks
        if i >= args.warmup:
            timed.append(last)
    seconds, voxels, tris = (sum(t[k] for t in timed) for k in range(3))
    value = voxels / seconds                                  # ratio of sums over the timed steps
    base = sample.describe(seconds, voxels, tris // len(timed), passes=len(timed))
    line = {"impl": "reference", "metric": "sdf_voxels_per_s_export_1024", "value": value, "unit": "voxels/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": seconds / len(timed) * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args), "cpu_baseline": base,
            "e2e": {"value": value, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_line(line)


def workload_config(args):
    return {"workload": "%s export, %d^3 cells (lattice %d^3), octree levels %d/%d/%d, %d gradient-descent steps, "
                        "256^3 bounding-box search" % (args.scene, 1 << args.level, (1 << args.level) + 1, args.level,
                                                        args.level, args.level, args.gd_steps),
            "voxels": "lattice cells covered by the export (cells per side cubed) per second -- the same rule in both arms; the "
                      "octree-ordered pass evaluates ~9 % of the lattice's samples (roofline_other.fraction_of_dense_lattice), like "
                      "the reference's walk, which culls whole subtrees",
            "scene": args.scene, "grid_level": args.level, "gd_steps": args.gd_steps,
            "parallelism": "z-slabs x%d" % args.gpus,
            "gather": "libdcsg communicator: NCCL all-reduce of the sharded search + all-gather of the slabs' counts; keys / triangles / "
                      "projected positions stored by the kernels into rank 0's arrays over NVLink (CUDA IPC peer mappings), no weld"
                      if args.gpus > 1 else None,
            "l2": "no flush: each step streams ~1.4 GB of bitmaps and mesh buffers, 11x the 126 MB L2"}


# ---------------------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path returned in its last step
# ---------------------------------------------------------------------------------------------------------------
DUMP_ROWS = 1 << 19                 # rows kept of a longer array; at most ~42 MB in all
DUMP_SEED = 20240601


def dump_outputs(out_dir, box, mesh, device):
    """Write the bounding box, the counts and the mesh's device arrays (projected vertex positions, vertex keys, triangles,
    active cells and their sign masks) as out_dir/<name>.npy, so that two builds can be compared output for output.

    An array longer than DUMP_ROWS keeps the rows np.random.default_rng(DUMP_SEED) draws from its length, sorted and saved
    as <group>_rows.npy (vertex_rows for vertices and vertex_keys, triangle_rows, cell_rows for cell_ids and cell_masks).
    Positions stay float32; ids, indices and masks are stored as float64, exact below 2^53.  For N > 1 the mesh is rank 0's
    gathered whole mesh, which holds no cell arrays: that dump has no cell_ids / cell_masks / cell_rows files."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    out = {"box": np.asarray(box, dtype=np.float64),
           "counts": np.array([mesh.num_vertices, mesh.num_triangles, mesh.num_cells], dtype=np.float64)}
    groups = (("vertex", mesh.num_vertices, ("vertices", "vertex_keys")), ("triangle", mesh.num_triangles, ("triangles",)),
              ("cell", mesh.num_cells, ("cell_ids", "cell_masks")))
    for group, n, names in groups:
        rows = np.arange(n)
        if n > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ROWS, replace=False))
            out[group + "_rows"] = rows.astype(np.float64)
        index = torch.from_numpy(rows).to(device)
        for name in names:
            view = mesh.device(name)
            if n and not view.__cuda_array_interface__["data"][0]:
                continue                                      # not kept by this path (e.g. cell arrays of a gathered mesh)
            picked = torch.as_tensor(view, device=device)[index].cpu().numpy() if n else np.zeros(0)
            out[name] = picked.astype(np.float32 if name == "vertices" else np.float64)
    total = sum(a.nbytes for a in out.values())
    assert total <= 64 << 20, total
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from designcsg_b200 import api, build, distributed as D
    from tests.golden import scenes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d: launch with torch.distributed.run for N > 1" % (args.gpus, world))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    build.build()
    scene = scenes.materialize(args.scene)
    ctx = api.Context(local)
    ctx.build(scene["dir"])
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    n_cells = 1 << args.level
    mesh = api.Mesh(ctx)
    device = torch.device("cuda", local)
    # N > 1: everything that crosses GPUs happens inside libdcsg (dcsg_comm: NCCL for the small collectives, peer stores for
    # the mesh); torch.distributed only carried the communicator id and reduces the timings at the end
    comm = D.create_comm(ctx) if world > 1 else None
    state = {}

    def step():
        if world == 1:
            box = ctx.bbox(SEARCH_DIAMETER)
            state["box"], state["slab"] = box, (0, n_cells)
            ctx.extract(box, args.level, gd_steps=args.gd_steps, copy_to_host=False, mesh=mesh)
            return
        # sharded 256^3 search (all-reduce of the extremes + the surface histogram) -> z-slabs balanced by that histogram (the
        # same plan on every rank) -> slab extraction; keys / triangles / projected positions are stored straight into rank
        # 0's arrays, which hold the whole mesh -- the single-GPU arrays -- when the call returns
        box = comm.bbox(SEARCH_DIAMETER)
        _, state["whole"], info = comm.extract(box, args.level, gd_steps=args.gd_steps, gather_to=0, mesh=mesh)
        state["box"], state["slab"], state["info"] = box, (info.slab_z0, info.slab_z1), info

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    fence()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    launches0 = api.launch_count()
    ctx.project_stats()                                    # clear the projection kernel's counters: the timed steps only
    stage_acc = {k: 0.0 for k in api.STAGES}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    with torch.cuda.stream(stream):
        ev0.record()
    for _ in range(args.steps):
        step()
        for k, v in mesh.stage_ms.items():
            stage_acc[k] += v
    with torch.cuda.stream(stream):
        ev1.record()
    fence()
    elapsed_ms = ev0.elapsed_time(ev1)
    launches = api.launch_count() - launches0
    tap_rounds, exact_rounds = (v / args.steps for v in ctx.project_stats())     # executed by the projection kernel, per step
    clock_info = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # before anything below reuses the mesh; for N > 1 rank 0's gathered arrays hold the whole mesh
        dump_outputs(args.dump_outputs, state["box"], mesh if world == 1 else state["whole"], device)
    if world > 1:
        t = torch.tensor([elapsed_ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
        info = state["info"]
        n_tris, n_verts, n_cells_active = int(info.total_triangles), int(info.total_vertices), int(info.total_cells)
        per_rank = [None] * world
        dist.all_gather_object(per_rank, {"slab": [int(info.slab_z0), int(info.slab_z1)], "triangles": mesh.num_triangles,
                                          "stage_ms": {k: round(v / args.steps, 4) for k, v in stage_acc.items()}})
    else:
        per_rank = None
        n_tris, n_verts, n_cells_active = mesh.num_triangles, mesh.num_vertices, mesh.num_cells
    slab = state["slab"]
    ms_per_step = elapsed_ms / args.steps
    voxels = float(n_cells) ** 3
    value = voxels / (ms_per_step * 1e-3)

    line = None
    if rank == 0:
        flop_eval = FLOP_PER_EVAL.get(args.scene)
        lattice_ms = stage_acc["lattice"] / args.steps
        project_ms = stage_acc["project"] / args.steps
        samples = float(mesh.c.lattice_samples)          # SDF evaluations of the (sparse) lattice stage on rank 0
        peak_fma = ctx.fp32_peak_tflops(0)
        peak_nofma = ctx.fp32_peak_tflops(1)

        def roof(kernel, flops, ms):
            achieved = flops / (ms * 1e-3) / 1e12 if flop_eval and ms > 0 else None
            return {"kernel": kernel, "bound": "fp32", "achieved": achieved, "peak": peak_fma, "unit": "TFLOP/s",
                    "frac": achieved / peak_fma if achieved else None,
                    "algorithmic_flop_per_evaluation": flop_eval,
                    "executed_flop_per_evaluation": EXECUTED_FLOP_PER_EVAL.get(args.scene) if kernel != "dcsg_k_lattice" else None,
                    "frac_executed": (achieved / peak_fma * EXECUTED_FLOP_PER_EVAL[args.scene] / flop_eval
                                      if achieved and args.scene in EXECUTED_FLOP_PER_EVAL and kernel != "dcsg_k_lattice" else None),
                    "peak_source": "measured in this run: FFMA micro-benchmark (dcsg_fp32_peak); FMUL/FADD-only issue rate "
                                   "%.1f TFLOP/s.  `achieved` counts the reference's operations (SURVEY.md 8d); the checked "
                                   "fast copy of the scene executes fewer of them (DESIGN.md 3b)" % peak_nofma,
                    "ms_per_launch": ms, "traffic": TRAFFIC.get(kernel)}

        proj_flops = float(mesh.num_vertices) * args.gd_steps * (7.0 * (flop_eval or 0) + FLOP_PER_NORMAL_EXTRA)
        r_lat = roof("dcsg_k_descend+dcsg_k_leaf+dcsg_k_corners", samples * (flop_eval or 0), lattice_ms)
        r_lat["evaluations"] = samples
        r_lat["fraction_of_dense_lattice"] = samples / (float((n_cells + 1) ** 2) * float(slab[1] - slab[0] + 1))
        # the dense lattice kernel (every sample of the slab), measured once outside the timed region
        dense_mesh = ctx.extract(state["box"], args.level, gd_steps=0, slab=slab, copy_to_host=False, dense=True)
        dense_mesh = ctx.extract(state["box"], args.level, gd_steps=0, slab=slab, copy_to_host=False, dense=True, mesh=dense_mesh)
        r_dense = roof("dcsg_k_lattice", float(dense_mesh.c.lattice_samples) * (flop_eval or 0), dense_mesh.stage_ms["lattice"])
        r_dense["evaluations"] = float(dense_mesh.c.lattice_samples)
        dense_mesh.free()
        # The projection kernel against the FFMA peak, three ways (DESIGN.md 5):
        #   frac                what it EXECUTED, charged at the reference's operation count: tap rounds counted by the kernel (a
        #                       vertex that reaches a fixed point stops early) x (7 evaluations x 287 + 22)
        #   frac_executed       the operations the instruction stream really holds: the checked fast copy runs 154 of the 287
        #                       per evaluation (zero-coefficient terms dropped), rounds repeated through the exact copy run 287
        #   frac_if_all_steps   SURVEY.md 8(d)'s formula, vertices x steps x (7 x 287 + 22), i.e. round 1's figure
        # plus the issue-slot utilisation ncu measured for this kernel (profiles/), the honest reading of an issue-bound kernel.
        r_proj = roof("dcsg_k_project", tap_rounds * (7.0 * (flop_eval or 0) + FLOP_PER_NORMAL_EXTRA), project_ms)
        r_proj["tap_rounds_executed"] = tap_rounds
        r_proj["tap_rounds_repeated_exactly"] = exact_rounds
        r_proj["tap_rounds_if_all_steps"] = float(mesh.num_vertices) * args.gd_steps
        if project_ms > 0 and flop_eval:
            r_proj["frac_if_all_steps"] = proj_flops / (project_ms * 1e-3) / 1e12 / peak_fma
            if args.scene in EXECUTED_FLOP_PER_EVAL:
                executed = tap_rounds * (7.0 * EXECUTED_FLOP_PER_EVAL[args.scene] + FLOP_PER_NORMAL_EXTRA) + exact_rounds * 7.0 * flop_eval
                r_proj["frac_executed"] = executed / (project_ms * 1e-3) / 1e12 / peak_fma
        r_proj["issue_active"] = TRAFFIC.get("dcsg_k_project.issue_active")
        # the list kernels of the mesher against HBM
        hbm_peak = None
        try:
            hbm_peak = float(json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))["hbm_gbs"])
            hbm_source = "MEASURED_PEAKS.json hbm_gbs"
        except (OSError, ValueError, KeyError):
            hbm_peak, hbm_source = 6534.0, "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"

        def hbm_roof(kernel, nbytes, ms, what):
            achieved = nbytes / (ms * 1e-3) / 1e9 if ms > 0 else None
            traffic = sum(TRAFFIC.get(k, 0.0) for k in kernel.split("+")) or None
            return {"kernel": kernel, "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak if achieved else None, "peak_source": hbm_source, "ms_per_launch": ms,
                    "algorithmic_bytes": nbytes, "algorithmic_bytes_formula": what, "traffic": traffic,
                    "traffic_over_algorithmic": traffic / nbytes if traffic and nbytes else None}

        # SURVEY.md 8(d)'s per-unit figures: classification + compaction = 4 B per lattice sample read + 4 B per active cell
        # (the lattice is never materialised here -- the pass keeps ONE BIT per evaluated sample -- so the samples are those the
        # octree-ordered pass evaluated); emission = 36 A + 12 U + 12 T.  Both stages are latency / integer-issue bound list
        # kernels, not HBM bound: the fractions say how far from the HBM roof they sit, `traffic` (ncu, per launch) how many
        # bytes they really moved.
        r_hbm = [hbm_roof("k_classify+k_worklist_count+k_worklist_fill+k_edges+k_scan_tiles", 4.0 * samples + 4.0 * mesh.num_cells,
                          stage_acc["classify"] / args.steps, "4 B x evaluated lattice samples + 4 B x active cells"),
                 hbm_roof("k_emit_vertices+k_emit_triangles", 36.0 * mesh.num_cells + 12.0 * mesh.num_vertices + 12.0 * mesh.num_triangles,
                          stage_acc["emit"] / args.steps, "36 A + 12 U + 12 T (active cells, unique vertices, triangles)")]
        dominant, other = (r_proj, r_lat) if project_ms >= lattice_ms else (r_lat, r_proj)
        line = {"metric": "sdf_voxels_per_s_export_1024", "value": value, "unit": "voxels/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(args), "clocks": clock_info, "gpu_launches": launches,
                "triangles": n_tris, "vertices": n_verts, "active_cells": n_cells_active,
                "triangles_per_s": n_tris / (ms_per_step * 1e-3),
                "stage_ms_rank0": {k: v / args.steps for k, v in stage_acc.items()}, "per_rank": per_rank,
                "slab_rank0": list(slab),
                "roofline": dominant, "roofline_other": other, "roofline_dense_lattice": r_dense, "roofline_hbm": r_hbm}

    # ---- e2e through the C ABI with HOST buffers -------------------------------------------------------------------
    # every step: side table host -> device, bounding-box search, (slab plan,) extraction + projection of this rank's
    # slab, then this rank's byte ranges of the byte-exact PLY + STL files device -> pinned host memory
    # (dcsg_format_segments).  For N > 1 the only communication is the all-gather of the triangle counts; the ranks'
    # segments concatenate to the single-GPU files (tests/test_gpu_parity.py::test_file_segments...).
    table = np.zeros(131072, dtype=np.float32)
    raw = open(os.path.join(scene["dir"], "arbitrary_data.hex"), "rb").read()
    table[:len(raw) // 4] = np.frombuffer(raw, dtype="<f4")

    def e2e_step():
        ctx.set_arbitrary_data(table)                                                   # H2D, every step
        if world == 1:
            box = ctx.bbox(SEARCH_DIAMETER)
            ctx.extract(box, args.level, gd_steps=args.gd_steps, copy_to_host=False, mesh=mesh, defer_projection=True)
            first = 0
        else:
            box = comm.bbox(SEARCH_DIAMETER)
            _, _, info = comm.extract(box, args.level, gd_steps=args.gd_steps, gather_to=-1, mesh=mesh, defer_projection=True)
            first = int(info.first_triangle)
        # projection in z-ordered chunks, each chunk's file rows formatted and copied (D2H, pinned) under the next one
        segs = mesh.project_and_format_segments(args.gd_steps, first)
        # segs = (PLY vertex rows, PLY face rows, STL records); the face rows (3, 3i, 3i+1, 3i+2 -- a function of the
        # triangle count alone) are written into the pinned buffer by host threads, the other two come over PCIe
        return segs[0].size + segs[2].size

    for _ in range(2):
        file_bytes = e2e_step()
    fence()
    t0 = time.perf_counter()
    e2e_steps = max(2, min(args.steps, 5))                # a secondary measurement with its own count: 2 to 5 steps
    for _ in range(e2e_steps):
        file_bytes = e2e_step()
    fence()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    io = torch.tensor([e2e_ms, float(file_bytes)], dtype=torch.float64, device=device)
    if world > 1:
        both = [torch.empty_like(io) for _ in range(world)]
        dist.all_gather(both, io)
        e2e_ms = max(float(b[0]) for b in both)
        file_bytes = int(sum(float(b[1]) for b in both))
    if rank == 0:
        line["e2e"] = {"value": voxels / (e2e_ms * 1e-3), "unit": "voxels/s", "ms_per_step": e2e_ms, "steps": e2e_steps,
                       "h2d_bytes_per_step": int((table.nbytes + 24) * world), "d2h_bytes_per_step": int(file_bytes + (12 + 24 + 8) * world),
                       "file_bytes_per_step": int(file_bytes / 122 * 135),
                       "what": "per rank: dcsg_set_arbitrary_data + dcsg_bbox[_sharded] + dcsg_extract[_sharded] + "
                               "dcsg_project_and_format_segments (projection pipelined with formatting and the D2H copies): the rank's "
                               "byte ranges of the byte-exact PLY + STL files in pinned host memory (vertex rows and STL records device -> host, "
                               "72 + 50 B per triangle; the 13 B face rows, which depend on the triangle count only, filled in by host threads) "
                               "(N > 1: sharded search all-reduce, all-gather of the slabs' counts); wall clock, max over ranks; disk write not included"}
    if world == 1:
        # file write, reported apart (page cache / disk dependent); the files go to a temporary directory, never the tree
        out_dir = tempfile.mkdtemp(prefix="dcsg_bench_")
        # the whole export INTO FILES (page cache / disk dependent, hence apart from e2e): search + extraction + projection
        # pipelined with formatting, D2H and the writes (dcsg_project_and_write_files)
        ply_path, stl_path = os.path.join(out_dir, "bench_export.ply"), os.path.join(out_dir, "bench_export.stl")
        to_files = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            box = ctx.bbox(SEARCH_DIAMETER)
            ctx.extract(box, args.level, gd_steps=args.gd_steps, copy_to_host=False, mesh=mesh, defer_projection=True)
            mesh.project_and_write_files(args.gd_steps, stl_path, ply_path)
            to_files.append((time.perf_counter() - t0) * 1e3)
        line["export_to_files_ms"] = min(to_files)
        t0 = time.perf_counter()
        mesh.write_ply(ply_path)
        mesh.write_stl(stl_path)
        line["write_ms"] = (time.perf_counter() - t0) * 1e3         # the two files written one after the other from a finished mesh
        shutil.rmtree(out_dir, ignore_errors=True)
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_reference_sample(args.scene, args.level, args.gd_steps, args.cpu_blocks)
    elif rank == 0:
        line["cpu_baseline"] = None

    if rank == 0:
        emit_line(line)
    mesh.free()
    if comm is not None:
        comm.barrier()
        comm.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def load_traffic():
    """dram bytes per launch from the committed ncu capture (profiles/traffic.json), or nothing."""
    path = os.path.join(REPO, "profiles", "traffic.json")
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except ValueError:
            pass
    return {}


TRAFFIC = load_traffic()


_REAL_STDOUT = None


def emit_line(line):
    """The ONE JSON line goes to the real stdout; everything else printed during the run (design scripts, NCCL's
    version banner, ...) was redirected to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                       # fd 1 -> stderr for libraries and child processes
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the main measurement; e2e times min(max(steps, 2), 5) steps of its own")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scene", default="design1")
    ap.add_argument("--level", type=int, default=10, help="grid level: 2^level cells per side")
    ap.add_argument("--gd-steps", type=int, default=50)
    ap.add_argument("--cpu-blocks", type=int, default=8, help="128^3 blocks in the CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
