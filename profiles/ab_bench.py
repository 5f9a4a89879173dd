"""A/B of builds of libqd_b200.so on one GPU: bench.py runs in turn with QD_B200_LIB set to each build.
    python profiles/ab_bench.py <out_dir> <lib_a> <lib_b> [<lib_c> ...] [--rounds 3] [-- bench.py arguments ...]
Each round runs every build once, in the order given (headline only: --no-extras --no-cpu-baseline --check-clips 0).
Then one more run per build with --dump-outputs, and each build's y.npy is compared bit for bit with the first one's
(the dumps are deleted afterwards).  Writes <out_dir>/ab.jsonl (one line per run, then one summary line per build:
median and spread, max - min, of `value` and of the spectral pass's ms per step) and prints the summary."""
import json
import os
import shutil
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench(lib, extra):
    env = dict(os.environ, QD_B200_LIB=os.path.abspath(lib))
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-extras", "--no-cpu-baseline",
           "--check-clips", "0"] + extra
    out = subprocess.run(cmd, env=env, check=True, capture_output=True, text=True).stdout
    return json.loads([ln for ln in out.splitlines() if ln.startswith("{")][-1])


def main():
    args = sys.argv[1:]
    extra = args[args.index("--") + 1:] if "--" in args else []
    args = args[:args.index("--")] if "--" in args else args
    rounds = 3
    if "--rounds" in args:
        i = args.index("--rounds")
        rounds = int(args[i + 1])
        del args[i:i + 2]
    out_dir, libs = args[0], args[1:]
    os.makedirs(out_dir, exist_ok=True)
    runs = {lib: [] for lib in libs}
    with open(os.path.join(out_dir, "ab.jsonl"), "w") as f:
        def emit(row):
            f.write(json.dumps(row) + "\n")
            f.flush()
            print(json.dumps(row), flush=True)

        for r in range(rounds):
            for lib in libs:
                res = bench(lib, extra)
                row = {"round": r, "lib": lib, "value": res["value"], "ms_per_step": res["ms_per_step"],
                       "spectral_ms_per_step": res["roofline"]["kernel_ms_per_step"]["spectral"], "clocks": res.get("clocks")}
                runs[lib].append(row)
                emit(row)
        dumps = []
        for i, lib in enumerate(libs):
            d = os.path.join(out_dir, f"dump_{i}")
            bench(lib, extra + ["--dump-outputs", d])
            dumps.append(np.load(os.path.join(d, "y.npy")))
            shutil.rmtree(d)
        for lib in libs:
            v = [r["value"] for r in runs[lib]]
            s = [r["spectral_ms_per_step"] for r in runs[lib]]
            emit({"lib": lib, "runs": len(v), "value_median": statistics.median(v), "value_spread": max(v) - min(v),
                  "spectral_ms_median": statistics.median(s), "spectral_ms_spread": max(s) - min(s)})
        for lib, y in zip(libs[1:], dumps[1:]):
            emit({"dump_vs_first": lib, "shape": list(y.shape), "array_equal": bool(np.array_equal(dumps[0], y)),
                  "bitwise_equal": bool(y.shape == dumps[0].shape and np.array_equal(dumps[0].view(np.uint32), y.view(np.uint32)))})


if __name__ == "__main__":
    main()
