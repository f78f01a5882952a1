"""A/B of two builds of the C-ABI library in one GPU session, selected through MDS_B200_LIB (e.g. a parent commit's library
built from a checkout of it, and this tree's).  Alternates the builds so that drift of the shared machine hits both:
  1. bench.py --gpus 1 --steps 100 --warmup 3 --no-cpu-baseline --no-e2e --no-strong, `reps` runs per build: value,
     C5_f64, C3_o2_16384, clocks;
  2. tools/variant_bench.py (single stream, 125 000 environments): ms per control step;
  3. bench.py --dump-outputs in fp32 and fp64: obs_log.npy / rollout_stats.npy compared byte for byte.
usage: python tools/ab_rollout.py <lib_a> <lib_b> <out_dir> [reps]     (one JSON summary line on stdout)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib_a, lib_b, out = os.path.abspath(sys.argv[1]), os.path.abspath(sys.argv[2]), os.path.abspath(sys.argv[3])
reps = int(sys.argv[4]) if len(sys.argv) > 4 else 3
os.makedirs(out, exist_ok=True)
LIBS = {"a": lib_a, "b": lib_b}
BENCH = ["--gpus", "1", "--steps", "100", "--warmup", "3", "--no-cpu-baseline", "--no-e2e", "--no-strong"]


def run(tag, args):
    env = dict(os.environ, MDS_B200_LIB=LIBS[tag])
    r = subprocess.run([sys.executable] + args, cwd=ROOT, env=env, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout[-2000:] + r.stderr[-4000:])
        raise SystemExit(f"{tag}: {' '.join(args)} failed ({r.returncode})")
    return r.stdout


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return r.stdout.strip()


res = {"card": card(), "libs": LIBS, "bench": {"a": [], "b": []}, "variant_ms_per_step": {"a": [], "b": []}}
for i in range(reps):
    for tag in ("a", "b") if i % 2 == 0 else ("b", "a"):
        line = [ln for ln in run(tag, ["bench.py"] + BENCH).splitlines() if ln.startswith("{")][-1]
        j = json.loads(line)
        with open(os.path.join(out, f"bench_{tag}_{i}.json"), "w") as f:
            f.write(line + "\n")
        cfg = j.get("configs", {})
        res["bench"][tag].append({"value": j.get("value"), "C5_f64": (cfg.get("C5_f64") or {}).get("value"),
                                  "C3_o2_16384": (cfg.get("C3_o2_16384") or {}).get("value"), "clocks": j.get("clocks")})
        print(tag, i, j.get("value"), file=sys.stderr, flush=True)
for i in range(reps):
    for tag in ("a", "b") if i % 2 == 0 else ("b", "a"):
        txt = run(tag, ["tools/variant_bench.py"])
        res["variant_ms_per_step"][tag].append(float(txt.split("ms/step")[1].split()[0]))
res["outputs_identical"] = {}
for dt in ("f32", "f64"):
    for tag in ("a", "b"):
        run(tag, ["bench.py", "--steps", "4", "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--no-strong", "--no-configs", "--dtype", dt,
                  "--dump-outputs", os.path.join(out, f"dump_{dt}_{tag}")])
    same = {}
    for name in sorted(os.listdir(os.path.join(out, f"dump_{dt}_a"))):
        with open(os.path.join(out, f"dump_{dt}_a", name), "rb") as fa, open(os.path.join(out, f"dump_{dt}_b", name), "rb") as fb:
            same[name] = fa.read() == fb.read()
    res["outputs_identical"][dt] = same
print(json.dumps(res))
