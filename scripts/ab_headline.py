"""A/B of the bench.py headline between built trees, in one process on one card.

    python scripts/ab_headline.py main=/path/to/main branch=/path/to/branch [--runs 5] [--out FILE.jsonl]

Each arm is LABEL=TREE, optionally followed by ,VAR=VALUE environment settings for that arm's processes
(e.g. branch=.,B2K_TPW_JAC=2).  The first arm is the reference.  Prints JSON lines:
  - the card: nvidia-smi name, power limit and max SM clock (read-only query);
  - one line per bench run: `bench.py --headline-only --no-cpu-baseline --dump-outputs`, arms interleaved
    A B A B ... so that drift on a shared host lands on every arm alike;
  - one summary per arm: median / min / max of ms_per_step and of step_ms.median, and whether its dumped
    T.npy / J.npy are byte-identical to the reference arm's;
  - scripts/kernel_bench.py --only probe_ (the HBM fill / copy ceiling) once, and --only fkine_jacob0
    (Panda / UR10, fp64 / fp32) per arm, interleaved, --kb-runs times.
"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np


def emit(d, fh):
    line = json.dumps(d)
    print(line, flush=True)
    if fh:
        fh.write(line + "\n")
        fh.flush()


def parse_arm(spec):
    label, _, rest = spec.partition("=")
    parts = rest.split(",")
    env = dict(p.split("=", 1) for p in parts[1:])
    return {"label": label, "tree": parts[0], "env": env}


def run_json(cmd, arm, timeout):
    env = dict(os.environ, **arm["env"])
    p = subprocess.run(cmd, cwd=os.path.abspath(arm["tree"]), env=env, capture_output=True, text=True, timeout=timeout)
    lines = []
    for ln in p.stdout.splitlines():
        ln = ln.strip()
        if ln.startswith("{"):
            try:
                lines.append(json.loads(ln))
            except json.JSONDecodeError:
                pass
    return p.returncode, lines, p.stderr[-2000:]


def digest(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest() if os.path.exists(path) else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("arms", nargs="+", help="LABEL=TREE[,VAR=VALUE...]; the first is the reference")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--kb-runs", type=int, default=2)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    arms = [parse_arm(s) for s in args.arms]
    if len(arms) < 2:
        ap.error("need at least two arms")
    dumps = tempfile.mkdtemp(prefix="ab_headline_")  # 30 MB per run: outside the trees and the output file
    fh = open(args.out, "w") if args.out else None

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    emit({"gpu": smi.stdout.strip(), "arms": {a["label"]: {"tree": a["tree"], "env": a["env"]} for a in arms}}, fh)

    runs = {a["label"]: [] for a in arms}
    sums = {a["label"]: [] for a in arms}
    for r in range(args.runs):
        for a in arms:
            d = os.path.join(dumps, f"{a['label']}_{r}")
            cmd = [sys.executable, "bench.py", "--headline-only", "--no-cpu-baseline", "--dump-outputs", d]
            rc, lines, err = run_json(cmd, a, 1200)
            res = next((x for x in lines if "ms_per_step" in x), None)
            if rc != 0 or res is None:
                emit({"arm": a["label"], "run": r, "rc": rc, "error": err}, fh)
                continue
            rec = {"arm": a["label"], "run": r, "ms_per_step": res["ms_per_step"],
                   "step_ms_median": res.get("step_ms", {}).get("median"), "parity": res.get("parity")}
            emit(rec, fh)
            runs[a["label"]].append(rec)
            sums[a["label"]].append((digest(os.path.join(d, "T.npy")), digest(os.path.join(d, "J.npy"))))

    ref = arms[0]["label"]
    ref_sums = set(sums[ref])
    for a in arms:
        rs = runs[a["label"]]
        if not rs:
            continue
        ms = np.array([x["ms_per_step"] for x in rs])
        sm = np.array([x["step_ms_median"] for x in rs if x["step_ms_median"] is not None])
        summ = {"summary": a["label"], "env": a["env"], "n": len(rs),
                "ms_per_step": {"median": float(np.median(ms)), "min": float(ms.min()), "max": float(ms.max())},
                "step_ms_median": {"median": float(np.median(sm)), "min": float(sm.min()), "max": float(sm.max())} if len(sm) else None,
                "outputs_identical_to_" + ref: len(set(sums[a["label"]])) == 1 and set(sums[a["label"]]) == ref_sums and len(ref_sums) == 1}
        if a["label"] != ref and runs[ref]:
            m0 = float(np.median([x["ms_per_step"] for x in runs[ref]]))
            summ["median_vs_" + ref] = float(np.median(ms)) / m0 - 1.0
            summ["slowest_faster_than_fastest_" + ref] = bool(ms.max() < min(x["ms_per_step"] for x in runs[ref]))
        emit(summ, fh)

    rc, lines, err = run_json([sys.executable, "scripts/kernel_bench.py", "--only", "probe_"], arms[0], 600)
    for x in lines:
        emit(dict(x, arm=arms[0]["label"]), fh)
    for r in range(args.kb_runs):
        for a in arms:
            rc, lines, err = run_json([sys.executable, "scripts/kernel_bench.py", "--only", "fkine_jacob0"], a, 900)
            if rc != 0:
                emit({"arm": a["label"], "kernel_bench_rc": rc, "error": err}, fh)
            for x in lines:
                emit(dict(x, arm=a["label"], run=r), fh)
    shutil.rmtree(dumps, ignore_errors=True)


if __name__ == "__main__":
    main()
