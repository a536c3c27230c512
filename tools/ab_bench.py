"""A/B/A/B runs of bench.py on ONE box (boxes of the pool differ by +-2 %, so two settings are only comparable when they
alternate on the same GPU).

    python tools/ab_bench.py --a "" --b "UB_MULTI_WGRAD=0" [--rounds 2] [--steps 20] [--gpus 1]

Each run is a fresh process (`bench.py --no-cpu-baseline`, UB_BENCH_U8=0 unless the setting says otherwise); prints one line per
run and the per-setting medians of ms/step (device-resident) and of the e2e ms/step.  Takes ~15 s per single-GPU run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(setting, steps, warmup, gpus, port):
    env = dict(os.environ, UB_BENCH_U8="0")
    for kv in setting.split():
        k, _, v = kv.partition("=")
        env[k] = v
    cmd = [sys.executable]
    if gpus > 1:
        cmd += ["-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={gpus}", "--master-addr", "127.0.0.1", "--master-port", str(port)]
    cmd += [os.path.join(ROOT, "bench.py"), "--gpus", str(gpus), "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline", "--no-eager-baseline"]
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    lines = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        raise SystemExit(f"bench failed for setting {setting!r}:\n{r.stderr[-2000:]}")
    return json.loads(lines[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--a", default="", help='environment of setting A, e.g. "UB_ASYNC_ZERO=1"')
    ap.add_argument("--b", required=True, help='environment of setting B, e.g. "UB_ASYNC_ZERO=0 UB_LIB_VARIANT=x"')
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--gpus", type=int, default=1)
    args = ap.parse_args()
    res = {"A": [], "B": []}
    port = 29600
    for r in range(args.rounds):
        for name, setting in (("A", args.a), ("B", args.b)):
            port += 1
            d = run(setting, args.steps, args.warmup, args.gpus, port)
            res[name].append(d)
            print(f"{name}{r} [{setting or 'default'}]: {d['ms_per_step']:.3f} ms/step  {d['value']:.1f} clips/s  e2e {d['e2e']['ms_per_step']:.3f} ms  "
                  f"loss {d['loss']}  sm {d['clocks']['sm_mhz']} MHz {d['clocks']['reasons']}", flush=True)
    for name, setting in (("A", args.a), ("B", args.b)):
        ms = statistics.median(d["ms_per_step"] for d in res[name])
        e2e = statistics.median(d["e2e"]["ms_per_step"] for d in res[name])
        print(f"median {name} [{setting or 'default'}]: {ms:.3f} ms/step, e2e {e2e:.3f} ms/step")
    a = statistics.median(d["ms_per_step"] for d in res["A"])
    b = statistics.median(d["ms_per_step"] for d in res["B"])
    print(f"B vs A: {100.0 * (a - b) / a:+.2f} % step time saved")


if __name__ == "__main__":
    main()
