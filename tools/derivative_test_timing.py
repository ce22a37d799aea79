"""Time the batched first-order derivative test (cplb_derivative_test_device) against the unfused alternative.

Three cases at 65,536 instances: 4-contact Ground (synthetic.ground_batch, seeded), 4-contact Superquadric, 8-contact Ground.
For each: the fused kernel (one CTA per instance, the perturbed points evaluated in shared memory) and the widened path (x widened
to N (n + 1) rows in torch, one cplb_eval_device of g + cost plus one of Jacobian + gradient at x, the differences and the
comparison in torch), both timed with CUDA events after warm-up, and their outputs compared bit for bit.  Prints the GPU name and
power limit with the numbers.  Needs a CUDA device (there is no CPU path to time).

    python tools/derivative_test_timing.py [--instances 65536] [--reps 10] [--out FILE]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import centroidalplanner_b200 as cpl  # noqa: E402
from centroidalplanner_b200 import synthetic  # noqa: E402
from helpers import configure  # noqa: E402
from test_gpu_derivative_test import KEYS, as_numpy, assert_same, widened  # noqa: E402

CASES = {"ground4": (synthetic.NAMES4, "ground", lambda N: synthetic.ground_batch(N, 4, 1002)),
         "superquadric4": (synthetic.NAMES4, "superquadric", lambda N: synthetic.superquadric_batch(N, 4, 1003)),
         "ground8": (synthetic.NAMES8, "ground", lambda N: synthetic.ground_batch(N, 8, 1004))}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return q.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception as e:  # noqa: BLE001
        return f"{torch.cuda.get_device_name()} (power limit not read: {e})"


def time_ms(fn, reps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--instances", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("derivative_test_timing.py needs a CUDA device")
    torch.cuda.set_device(0)
    lines = [f"GPU: {gpu_info()}", f"instances: {a.instances}, timed repetitions per path: {a.reps} (after 2 warm-up calls), CUDA events",
             f"{'case':<15}{'n':>5}{'m':>5}{'fused ms':>12}{'widened ms':>12}{'widened/fused':>15}  outputs"]
    for name, (names, env_name, gen) in CASES.items():
        env = {"ground": cpl.Ground, "superquadric": cpl.Superquadric}[env_name]()
        prob = cpl.BatchedCplProblem(names, 100.0, env)
        configure(prob, env, names, env_name)
        x = torch.as_tensor(gen(a.instances), device="cuda")
        for _ in range(2):
            fused = prob.DerivativeTest(x)
            ref = widened(prob, x)
        torch.cuda.synchronize()
        assert_same(as_numpy(fused), as_numpy(ref), name)
        t_fused = time_ms(lambda: prob.DerivativeTest(x), a.reps)
        t_wide = time_ms(lambda: widened(prob, x), a.reps)
        del ref
        torch.cuda.empty_cache()
        lines.append(f"{name:<15}{prob.n:>5}{prob.m:>5}{t_fused:>12.3f}{t_wide:>12.3f}{t_wide / t_fused:>15.2f}  identical ({len(KEYS)} outputs)")
        print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
