"""A/B timing of two built trees on the benchmark workloads, alternating them, plus an output comparison.

  python tools/wf_payload_ab.py --base DIR [--new DIR] --out DIR [--reps 3] [--steps 20]

DIR is a repository tree whose libraries are built.  For each repetition the default workload runs once from --base,
then once from --new (default: this tree); the first run of each tree also dumps its image.  Then the two synthetic
GI workloads run once per tree, with their outputs dumped.  The dumps go to a temporary directory, removed at the end.
Every bench.py JSON line is written to <out>/bench_lines.jsonl with its tree and run; a table of the fields that
matter for the wavefront pipeline, the card's name and power limit (nvidia-smi query), and whether the dumped outputs
are byte-identical go to stdout."""
import argparse
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QUICK = ["--no-cpu-baseline", "--no-ref-cuda", "--no-cull", "--no-lbvh", "--no-protocol"]


def bench(tree, workload, steps, warmup, dump):
    cmd = [sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup",
           str(warmup), "--workload", workload] + QUICK
    if dump:
        cmd += ["--dump-outputs", dump]
    out = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
    if out.returncode != 0:
        sys.stderr.write(out.stdout[-4000:] + out.stderr[-4000:])
        raise SystemExit("bench.py failed in %s (%s)" % (tree, workload))
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    return json.loads(lines[-1])


def fields(res):
    roof = res.get("roofline", {})
    k = roof.get("kernels", {})
    return {"ms_per_step": res.get("ms_per_step"),
            "k_wf_shade_ms": k.get("k_wf_shade", {}).get("ms_per_step"),
            "k_wf_primary_ms": k.get("k_wf_primary", {}).get("ms_per_step"),
            "traversal_ms": roof.get("traversal_ms_per_step"),
            "clocks": res.get("clocks")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=True)
    ap.add_argument("--new", default=ROOT)
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    trees = {"base": os.path.abspath(args.base), "new": os.path.abspath(args.new)}
    out = os.path.abspath(args.out)
    os.makedirs(out, exist_ok=True)
    dumps = tempfile.mkdtemp(prefix="wf_ab_")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout
    print(smi.strip())
    log = open(os.path.join(out, "bench_lines.jsonl"), "w")
    runs = []
    for rep in range(args.reps):
        for tag, tree in trees.items():
            dump = os.path.join(dumps, tag, "cornell_gi_1080p_64spp") if rep == 0 else None
            res = bench(tree, "cornell_gi_1080p_64spp", args.steps, 3, dump)
            log.write(json.dumps({"tree": tag, "rep": rep, "workload": "cornell_gi_1080p_64spp", "line": res}) + "\n")
            log.flush()
            runs.append((tag, rep, "cornell_gi_1080p_64spp", fields(res)))
            print(tag, rep, json.dumps(runs[-1][3]), flush=True)
    for workload, steps in (("synth1m_gi_1080p_16spp", 10), ("synth5m_gi_4k_256spp", 2)):
        for tag, tree in trees.items():
            res = bench(tree, workload, steps, 1, os.path.join(dumps, tag, workload))
            log.write(json.dumps({"tree": tag, "rep": 0, "workload": workload, "line": res}) + "\n")
            log.flush()
            runs.append((tag, 0, workload, fields(res)))
            print(tag, workload, json.dumps(runs[-1][3]), flush=True)
    for workload in ("cornell_gi_1080p_64spp", "synth1m_gi_1080p_16spp", "synth5m_gi_4k_256spp"):
        a, b = os.path.join(dumps, "base", workload), os.path.join(dumps, "new", workload)
        names = sorted(os.listdir(a))
        same = names == sorted(os.listdir(b)) and all(filecmp.cmp(os.path.join(a, n), os.path.join(b, n), shallow=False)
                                                     for n in names)
        print("outputs %s: %s %s" % (workload, names, "byte-identical" if same else "DIFFER"))
    shutil.rmtree(dumps)
    for tag in trees:
        ms = [f["ms_per_step"] for t, _, w, f in runs if t == tag and w == "cornell_gi_1080p_64spp"]
        sh = [f["k_wf_shade_ms"] for t, _, w, f in runs if t == tag and w == "cornell_gi_1080p_64spp"]
        print("%s default: ms_per_step %.3f-%.3f (spread %.3f), k_wf_shade %.3f-%.3f ms"
              % (tag, min(ms), max(ms), max(ms) - min(ms), min(sh), max(sh)))


if __name__ == "__main__":
    main()
