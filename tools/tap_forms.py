"""Developer timing loop: the two tap forms of the checked fast copy (DCSG_TAP_FORM=loop / axis, DESIGN.md 3b) built side by
side in one process and timed alternately on one GPU -- one extraction + projection of the whole mesh per run.
python tools/tap_forms.py SCENE LEVEL RUNS [OUT.json]"""
import json, os, statistics, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from designcsg_b200 import api, build
from tests.golden import scenes

build.build()
name, level, runs = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                     stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
scene_dir = scenes.materialize(name)["dir"]
forms = ("loop", "axis")
ctxs, logs = {}, {}
for form in forms:
    os.environ["DCSG_TAP_FORM"] = form          # read when the scene is compiled (dcsg_build)
    ctxs[form] = api.Context(0)
    logs[form] = ctxs[form].build(scene_dir)
os.environ.pop("DCSG_TAP_FORM")
box = ctxs["loop"].bbox(10.0)
meshes = {form: None for form in forms}
samples = {form: {"project": [], "step": []} for form in forms}
stats = {}
for rep in range(runs + 1):                     # run 0 of each form is the warm-up
    for form in (forms if rep % 2 == 0 else forms[::-1]):
        ctx = ctxs[form]
        ctx.project_stats()
        meshes[form] = ctx.extract(box, level, gd_steps=50, copy_to_host=False, mesh=meshes[form])
        st = meshes[form].stage_ms
        stats[form] = ctx.project_stats()
        if rep:
            samples[form]["project"].append(st["project"])
            samples[form]["step"].append(sum(v for k, v in st.items() if k != "copy"))
out = {"scene": name, "level": level, "runs": runs, "gpu": gpu, "project_stats": stats,
       "logs": {f: [l for l in (logs[f] or "").splitlines() if l.startswith("[dcsg]")] for f in forms}}
for form in forms:
    for key, vals in samples[form].items():
        out["%s_%s_ms" % (form, key)] = {"median": statistics.median(vals), "min": min(vals), "max": max(vals), "all": vals}
print(json.dumps(out, indent=1))
if len(sys.argv) > 4:
    with open(sys.argv[4], "w") as f:
        json.dump(out, f, indent=1)
for form in forms:
    meshes[form].free()
    ctxs[form].close()
