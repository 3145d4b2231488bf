"""The sharded export drivers on a one-rank communicator, against the single-GPU exports."""
import pytest

from tests.golden import scenes

pytestmark = pytest.mark.gpu


def test_sharded_export_on_one_rank_is_the_single_gpu_export(libdcsg, tmp_path):
    """dcsg_export_sharded and dcsg_export_sharded_indexed on a one-rank communicator write the files of dcsg_export and
    dcsg_export_indexed byte for byte, with the same progress states and report; adaptive levels stay refused for the sharded
    indexed export.  On a one-GPU machine this is what runs the sharded export drivers."""
    # torch first, as in every process that drives a communicator from Python: libdcsg then uses the NCCL torch loaded.  Loaded
    # the other way round, the NCCL libdcsg finds would stay in place and a later torch import in this process could fail.
    import torch  # noqa: F401
    from designcsg_b200 import api
    try:
        uid = api.comm_unique_id()
    except api.DcsgError as e:
        if e.code != -7:
            raise
        pytest.skip("NCCL is not loadable: %s" % e)
    scene = scenes.materialize("design1")["dir"]
    ctx = api.Context(0)
    comm = api.Comm(ctx, uid, 0, 1)
    try:
        seen = []
        cb = api.PROGRESS_FN(lambda user, state, done, total: seen.append((state, done, total)))
        ctx.set_progress_callback(cb)

        def run(fn, *args, **kwargs):
            del seen[:]
            rep = fn(*args, **kwargs)
            return rep, list(seen)

        def same_run(one, world1):
            (r1, p1), (rw, pw) = one, world1
            assert p1 == pw and p1[-1][0] == api.PROGRESS_STATES.index("COMPLETE")
            assert (r1.num_vertices, r1.num_triangles, r1.num_cells) == (rw.num_vertices, rw.num_triangles, rw.num_cells)
            assert r1.num_triangles > 0 and list(r1.box) == list(rw.box)

        for level in (7, 0):                # 0: the design's shipped octree levels (adaptive walk + retopologize)
            one = run(ctx.export, scene, level, str(tmp_path / "1.stl"), str(tmp_path / "1.ply"))
            world1 = run(comm.export, scene, level, str(tmp_path / "w.stl"), str(tmp_path / "w.ply"))
            same_run(one, world1)
            for ext in ("stl", "ply"):
                assert (tmp_path / ("1." + ext)).read_bytes() == (tmp_path / ("w." + ext)).read_bytes(), (level, ext)
        for normals in (False, True):
            one = run(ctx.export_indexed, scene, 7, str(tmp_path / "1i.ply"), normals=normals)
            world1 = run(comm.export_indexed, scene, 7, str(tmp_path / "wi.ply"), normals=normals)
            same_run(one, world1)
            assert (tmp_path / "1i.ply").read_bytes() == (tmp_path / "wi.ply").read_bytes(), normals
        with pytest.raises(api.DcsgError) as err:
            comm.export_indexed(scene, 0, str(tmp_path / "a.ply"))
        assert err.value.code == -7
        ctx.set_progress_callback(None)
    finally:
        comm.close()
        ctx.close()
