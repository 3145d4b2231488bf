"""Multi-GPU check of the indexed PLY, run under torchrun (tests/test_indexed_export.py::test_sharded_indexed_on_two_gpus):
dcsg_export_sharded_indexed gives the bytes of the single-GPU dcsg_export_indexed file for uniform levels 7 and 9 (with and
without normals), and the design's adaptive levels return DCSG_ERR_UNSUPPORTED on every rank without a hang."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from designcsg_b200 import api, build, distributed as D      # noqa: E402
from tests.golden import scenes                              # noqa: E402

out_dir = sys.argv[1]
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
build.build()

scene = scenes.materialize("design1")["dir"]
ctx = api.Context(local)
ctx.build(scene)
comm = D.create_comm(ctx)
for level in (7, 9):
    for normals in (False, True):
        sharded = os.path.join(out_dir, "sharded_%d_%d.ply" % (level, normals))
        rep = comm.export_indexed(scene, level, sharded, normals=normals)
        if rank == 0:
            single = os.path.join(out_dir, "single_%d_%d.ply" % (level, normals))
            ctx.export_indexed(scene, level, single, normals=normals)
            a, b = open(sharded, "rb").read(), open(single, "rb").read()
            assert a == b, "level %d normals %d: sharded file differs from the single-GPU file (%d vs %d bytes)" % (level, normals, len(a), len(b))
            print("indexed[design1 level %d, normals %d, %d GPUs]: %d vertices, %d triangles, %d bytes: BYTE-EQUAL to one GPU"
                  % (level, normals, world, rep.num_vertices, rep.num_triangles, len(a)))
            os.remove(single)
        comm.barrier()
        if rank == 0:
            os.remove(sharded)
try:
    comm.export_indexed(scene, 0, os.path.join(out_dir, "adaptive.ply"))
    raise SystemExit("rank %d: the adaptive levels were not refused" % rank)
except api.DcsgError as e:
    assert e.code == -7, e          # DCSG_ERR_UNSUPPORTED
comm.barrier()                      # every rank got here: nobody waits in a collective the others skipped
comm.close()
ctx.close()
dist.destroy_process_group()
if rank == 0:
    print("INDEXED MULTI-GPU OK")
