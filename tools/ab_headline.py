"""A/B of the headline benchmark between two builds of libkfb200.so, alternated in one session (dev tool).

    python tools/ab_headline.py --lib-a build/variants/libkfb200_parent.so --out DIR [--runs 3]

Build A is selected with KFB_LIB; build B is the in-tree library.  Records the card's name and power limit, then:
  1. runs `bench.py --dump-outputs` once per build and compares logp.npy, grad.npy and c5_*.npy byte for byte;
  2. alternates `bench.py --no-cpu-baseline` A, B, A, B, ... --runs times each and keeps every JSON result line.
Everything goes to DIR/ab_headline.json (and the dumps to DIR/dump_a, DIR/dump_b)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench(lib, extra):
    env = dict(os.environ)
    env.pop("KFB_LIB", None)
    if lib:
        env["KFB_LIB"] = os.path.abspath(lib)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1"] + extra, cwd=ROOT, env=env,
                       capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError(f"bench.py failed ({p.returncode}):\n{p.stderr[-4000:]}")
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    return json.loads(lines[-1])


def pick(r):
    # "roofline" is whichever of the two kernels took longer, "roofline_<other>" the other one: key them by kernel
    launch = {}
    for k in ("roofline", "roofline_adjoint", "roofline_forward"):
        if k in r:
            launch["adjoint" if r[k]["kernel"].startswith("kf_p1_adjoint") else "forward"] = r[k]["ms_per_launch"]
    c5 = r.get("c5") or {}
    return {"ms_per_step": r.get("ms_per_step"), "value": r.get("value"), "ms_per_launch": launch,
            "c5_ms_per_step": c5.get("ms_per_step"), "c5_value": c5.get("value"),
            "c5_draws_with_info": c5.get("draws_with_info"),
            "e2e_ms_per_step": r.get("e2e", {}).get("ms_per_step"),
            "draws_with_info": r.get("config", {}).get("draws_with_info")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib-a", required=True, help="library of build A (the parent)")
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    res = {"gpu": smi, "lib_a": a.lib_a, "lib_b": "in-tree", "dump": {}, "runs": []}
    import numpy as np

    dirs = {}
    for tag, lib in (("a", a.lib_a), ("b", None)):
        dirs[tag] = os.path.join(os.path.abspath(a.out), "dump_" + tag)
        bench(lib, ["--no-cpu-baseline", "--steps", "20", "--warmup", "3", "--dump-outputs", dirs[tag]])
    for f in sorted(os.listdir(dirs["a"])):
        if f.endswith(".npy"):
            x, y = np.load(os.path.join(dirs["a"], f)), np.load(os.path.join(dirs["b"], f))
            same = x.shape == y.shape and x.tobytes() == y.tobytes()
            diff = None if same or x.shape != y.shape else {
                "values_differing": int((x != y).sum()), "max_abs": float(np.nanmax(np.abs(x - y)))}
            res["dump"][f] = {"identical": same, "diff": diff}
    for i in range(a.runs):
        for tag, lib in (("a", a.lib_a), ("b", None)):
            r = bench(lib, ["--no-cpu-baseline"])
            res["runs"].append({"build": tag, "pair": i, "summary": pick(r), "result": r})
            print(tag, i, json.dumps(pick(r)), flush=True)
    with open(os.path.join(a.out, "ab_headline.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print("gpu:", smi)
    print("dump:", json.dumps(res["dump"]))
    for i in range(a.runs):
        ra, rb = (next(x for x in res["runs"] if x["build"] == t and x["pair"] == i)["summary"] for t in "ab")
        print(f"pair {i}: A {ra['ms_per_step']:.4f} ms  B {rb['ms_per_step']:.4f} ms  "
              f"({100 * (1 - rb['ms_per_step'] / ra['ms_per_step']):.1f} % less)  launches {ra['ms_per_launch']} -> "
              f"{rb['ms_per_launch']}")


if __name__ == "__main__":
    main()
