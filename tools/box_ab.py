#!/usr/bin/env python
"""A/B of the streaming box kernel against the library of another revision, in one run on one GPU.

  python tools/box_ab.py prepare [REV]     (no GPU needed) compile REV's library (default HEAD~1) into build/box_ab/<rev>/
  python tools/box_ab.py run [--runs N] [--out DIR]

`run` alternates, A B A B ..., N times each (default 5):
  bench.py --gpus 1 --no-extras --cpu-budget 0.5   on this tree (A) and on a temporary copy of it whose vpp_b200/lib/libvppb.so
                                                    is the prepared library (B),
  tools/box_bench.py's child                        on the same two trees (its batched 4K and 8K rows run the same kernel).
Each bench run records value, roofline.frac and clocks, with the GPU name and power limit read by `nvidia-smi --query-gpu`
right before it.  The first run of each side also passes --dump-outputs; the two dumps must be identical byte for byte.
Writes DIR/box_ab.json (default build/box_ab/result) and prints a markdown table."""
import argparse
import filecmp
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PREP = os.path.join(ROOT, "build", "box_ab")


def prepare(rev):
    sha = subprocess.check_output(["git", "-C", ROOT, "rev-parse", "--short", rev], text=True).strip()
    dst = os.path.join(PREP, sha)
    src = os.path.join(dst, "src")
    shutil.rmtree(dst, ignore_errors=True)
    os.makedirs(src)
    arch = subprocess.run(["git", "-C", ROOT, "archive", sha, "vpp_b200/csrc", "include"], check=True, capture_output=True).stdout
    subprocess.run(["tar", "-x", "-C", src], input=arch, check=True)
    cus = sorted(os.path.join(src, "vpp_b200", "csrc", f) for f in os.listdir(os.path.join(src, "vpp_b200", "csrc")) if f.endswith(".cu"))
    # the compile line of build.sh
    subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++14", "-fmad=false", "-Xcompiler", "-fPIC",
                    "-shared", "-o", os.path.join(dst, "libvppb.so")] + cus + ["-ldl"], check=True)
    shutil.rmtree(src)
    with open(os.path.join(PREP, "rev"), "w") as f:
        f.write(sha)
    print("prepared", os.path.join(dst, "libvppb.so"))


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        line = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else ""
    except OSError:
        line = ""
    name, _, power = line.partition(",")
    return {"name": name.strip(), "power_limit": power.strip()}


def bench(tree, dump_dir):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--no-extras", "--cpu-budget", "0.5"] + (["--dump-outputs", dump_dir] if dump_dir else [])
    info = gpu_info()
    r = subprocess.run(cmd, cwd=tree, capture_output=True, text=True, timeout=900)
    if r.returncode != 0:
        return dict(info, error=(r.stderr or r.stdout)[-2000:])
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    return dict(info, value=line["value"], frac=line["roofline"]["frac"], us_per_launch=line["roofline"]["us_per_launch"],
                clocks=line.get("clocks"), parity_checked=line.get("parity_checked"))


def box_rows(tree):
    info = gpu_info()
    r = subprocess.run([sys.executable, os.path.join("tools", "box_bench.py"), "child"], cwd=tree, capture_output=True, text=True, timeout=900)
    if r.returncode != 0:
        return dict(info, error=(r.stderr or r.stdout)[-2000:])
    rows = json.loads(r.stdout.strip().splitlines()[-1])
    return dict(info, rows={k: v for k, v in rows.items() if k.startswith("batch")})


def run(args):
    rev = open(os.path.join(PREP, "rev")).read().strip()
    lib_b = os.path.join(PREP, rev, "libvppb.so")
    out = os.path.abspath(args.out)
    os.makedirs(out, exist_ok=True)
    tmp = tempfile.mkdtemp(prefix="box_ab_")
    tree_b = os.path.join(tmp, "tree")
    shutil.copytree(ROOT, tree_b, symlinks=True, ignore=shutil.ignore_patterns(".git", "build", "__pycache__"))
    shutil.copy2(lib_b, os.path.join(tree_b, "vpp_b200", "lib", "libvppb.so"))
    sides = {"A": ROOT, "B": tree_b}
    res = {"B_rev": rev, "runs": {"A": [], "B": []}, "box_bench": {"A": [], "B": []}}
    try:
        for i in range(args.runs):
            for s in ("A", "B"):
                dump = os.path.join(tmp, "dump_" + s) if i == 0 else None
                res["runs"][s].append(bench(sides[s], dump))
                print(s, i, json.dumps(res["runs"][s][-1]), file=sys.stderr, flush=True)
        for i in range(args.box_runs):
            for s in ("A", "B"):
                res["box_bench"][s].append(box_rows(sides[s]))
                print("box_bench", s, i, json.dumps(res["box_bench"][s][-1]), file=sys.stderr, flush=True)
        fa, fb = os.path.join(tmp, "dump_A", "box5x5.npy"), os.path.join(tmp, "dump_B", "box5x5.npy")
        res["outputs_identical"] = os.path.exists(fa) and os.path.exists(fb) and filecmp.cmp(fa, fb, shallow=False)
        res["dump_bytes"] = os.path.getsize(fa) if os.path.exists(fa) else None
    finally:
        shutil.rmtree(tmp, ignore_errors=True)

    va = [r["value"] for r in res["runs"]["A"] if "value" in r]
    vb = [r["value"] for r in res["runs"]["B"] if "value" in r]
    if va and vb:
        res["median_A"], res["median_B"] = statistics.median(va), statistics.median(vb)
        res["speedup_median"] = res["median_A"] / res["median_B"]
        res["every_A_faster_than_every_B"] = min(va) > max(vb)
    with open(os.path.join(out, "box_ab.json"), "w") as f:
        json.dump(res, f, indent=1)

    print("| run | side | GPU | power limit | Mpix/s | frac of measured peak | us/launch | SM MHz (max) | throttle |")
    print("|---|---|---|---|---|---|---|---|---|")
    for i in range(args.runs):
        for s in ("A", "B"):
            r = res["runs"][s][i]
            if "value" not in r:
                print("| %d | %s | %s | %s | error | | | | |" % (i, s, r["name"], r["power_limit"]))
                continue
            c = r.get("clocks") or {}
            print("| %d | %s | %s | %s | %.0f | %.3f | %.1f | %s (%s) | %s |" % (i, s, r["name"], r["power_limit"], r["value"], r["frac"], r["us_per_launch"],
                                                                     c.get("sm_mhz"), c.get("sm_max_mhz"), ",".join(c.get("reasons") or [])))
    for s in ("A", "B"):
        for r in res["box_bench"][s]:
            print("box_bench %s: %s" % (s, json.dumps(r.get("rows", r.get("error")))))
    print(json.dumps({k: res.get(k) for k in ("B_rev", "median_A", "median_B", "speedup_median", "every_A_faster_than_every_B", "outputs_identical")}))


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    sub = ap.add_subparsers(dest="cmd", required=True)
    p = sub.add_parser("prepare")
    p.add_argument("rev", nargs="?", default="HEAD~1")
    r = sub.add_parser("run")
    r.add_argument("--runs", type=int, default=5)
    r.add_argument("--box-runs", type=int, default=3)
    r.add_argument("--out", default=os.path.join(PREP, "result"))
    a = ap.parse_args()
    prepare(a.rev) if a.cmd == "prepare" else run(a)
