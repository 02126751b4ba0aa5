"""Run bench.py (device-resident leg only) once per value of an environment variable and print the stage split.
usage: python tools/env_sweep.py VAR v1 v2 ... [-- extra bench args]
("-" leaves VAR unset), e.g. this build against another one: python tools/env_sweep.py LANE_B200_LIB - OTHER/liblane_b200.so"""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
args = sys.argv[1:]
extra = []
if "--" in args:
    i = args.index("--"); extra = args[i + 1:]; args = args[:i]
var, values = args[0], args[1:]
for v in values:
    env = dict(os.environ)
    if v != "-": env[var] = v
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "20", "--warmup", "3", "--skip-cpu",
                          "--skip-e2e"] + extra, env=env, capture_output=True, text=True)
    try:
        d = json.loads(out.stdout.strip().splitlines()[-1])
        s = d["stage_ms_per_step"]
        print(f"{var}={v}: value={d['value']:.0f} ms/step={d['ms_per_step']:.3f} k1={s['blur_hist']:.4f} canny={s['canny']:.4f} "
              f"ppht={s['ppht']:.4f} fit={s['fit']:.4f} frac={d['roofline']['frac']:.3f}", flush=True)
    except Exception as e:
        print(f"{var}={v}: FAILED {e} {out.stderr[-500:]}", flush=True)
