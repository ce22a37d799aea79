"""Time the fused Jacobian products (cplb_jacobian_products_device) against the materialising path.

Cases: 4-contact Ground, 4-contact Superquadric and 8-contact Ground (seeded synthetic batches), at 65,536 and 1,048,576 instances.
For each, both products:
  reverse  x_bar = obj_factor * grad f + J^T lambda
  forward  g_dot = J v,  f_dot = grad f . v
by two paths:
  fused          one cplb_jacobian_products_device call;
  materialising  cplb_eval_device for J and the gradient, then the products in torch: the factors gathered by iRow / jCol as
                 lockstep_solver.py gathers them, each sum taken in slot order (one gather, multiply and add per position of a
                 padded per-column / per-row slot table), which is the order of the bit contract, so the two paths' outputs are
                 compared bit for bit.
A third time is given for reference: the same products with lockstep_solver.py's index_add (its sums run in atomic order, so its
bits are not compared).  Times are CUDA events over --reps calls after 2 warm-up calls.  The algorithmic bytes per instance are
what a product has to move at least: x, the factors and the results, 8 (2n + m + 1) bytes either way.  Prints the GPU name and
power limit with the numbers.  Needs a CUDA device (there is no CPU path to time).

    python tools/jacobian_products_timing.py [--instances 65536 1048576] [--reps 20] [--out FILE]
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

HBM_GBS = 6449.7  # measured copy bandwidth of the B200 (DESIGN.md §4)
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


def slot_table(index, count):
    """(count, R) slots of each target (column or row), ascending, padded with -1."""
    index = index.cpu()
    R = int(torch.bincount(index, minlength=count).max())
    table = torch.full((count, R), -1, dtype=torch.int64)
    fill = [0] * count
    for s, t in enumerate(index.tolist()):
        table[t, fill[t]] = s
        fill[t] += 1
    return table


class Materialising:
    """cplb_eval_device's J and gradient, then the products summed in slot order."""

    def __init__(self, prob, iRow, jCol):
        self.prob, self.iRow, self.jCol = prob, iRow, jCol
        dev = iRow.device
        self.by_col = slot_table(jCol, prob.n).to(dev)
        self.by_row = slot_table(iRow, prob.m).to(dev)
        self.cols = torch.arange(prob.n, device=dev)

    @staticmethod
    def ordered(acc, vals, fac, other, table):
        """acc[:, t] + vals[:, s] * fac[:, other[s]] for the slots s of table row t, in table order."""
        for r in range(table.shape[1]):
            s = table[:, r]
            valid = s >= 0
            s = s.clamp(min=0)
            acc = torch.where(valid, acc + vals[:, s] * fac[:, other[s]], acc)
        return acc

    def __call__(self, x, lam=None, obj=None, v=None):
        p = self.prob
        ev = p.eval(x, g=False, jac=True, cost=False, grad=True)
        jac, grad = ev["jac"], ev["grad"]
        if v is None:
            return {"x_bar": self.ordered(obj[:, None] * grad, jac, lam, self.iRow, self.by_col)}
        zeros = lambda k: torch.zeros(x.shape[0], k, dtype=torch.float64, device=x.device)  # noqa: E731
        return {"g_dot": self.ordered(zeros(p.m), jac, v, self.jCol, self.by_row),
                "f_dot": self.ordered(zeros(1), grad, v, self.cols, self.cols[None, :])[:, 0]}

    def index_add(self, x, lam=None, obj=None, v=None):
        """lockstep_solver.py's gather / index_add (timed only)."""
        p = self.prob
        ev = p.eval(x, g=False, jac=True, cost=False, grad=True)
        jac, grad = ev["jac"], ev["grad"]
        if v is None:
            return (obj[:, None] * grad).index_add(1, self.jCol, jac * lam[:, self.iRow])
        return torch.zeros(x.shape[0], p.m, dtype=torch.float64, device=x.device).index_add(1, self.iRow, jac * v[:, self.jCol]), (grad * v).sum(1)


def identical(a, b):
    return all(bool(((a[k].view(torch.int64) == b[k].view(torch.int64)) | (a[k].isnan() & b[k].isnan())).all()) for k in a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--instances", type=int, nargs="+", default=[65536, 1048576])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("jacobian_products_timing.py needs a CUDA device")
    torch.cuda.set_device(0)
    lines = [f"GPU: {gpu_info()}", f"timed repetitions per path: {a.reps} (after 2 warm-up calls), CUDA events; "
             f"algorithmic bytes 8 (2n + m + 1) per instance, share of the measured {HBM_GBS} GB/s",
             f"{'case':<15}{'N':>9}{'mode':>9}{'B/inst':>8}{'fused ms':>10}{'GB/s':>8}{'of HBM':>8}{'mat. ms':>10}{'mat/fused':>10}"
             f"{'index_add ms':>14}  identical"]
    for name, (names, env_name, gen) in CASES.items():
        env = {"ground": cpl.Ground, "superquadric": cpl.Superquadric}[env_name]()
        prob = cpl.BatchedCplProblem(names, 100.0, env)
        configure(prob, env, names, env_name)
        iRow, jCol = (torch.as_tensor(t, dtype=torch.int64, device="cuda") for t in prob.GetJacobianStructure())
        mat_path = Materialising(prob, iRow, jCol)
        for N in a.instances:
            x = torch.as_tensor(gen(N), device="cuda")
            gen_ = torch.Generator(device="cuda").manual_seed(N)
            lam = torch.randn(N, prob.m, dtype=torch.float64, device="cuda", generator=gen_)
            obj = torch.rand(N, dtype=torch.float64, device="cuda", generator=gen_)
            v = torch.randn(N, prob.n, dtype=torch.float64, device="cuda", generator=gen_)
            bytes_inst = 8 * (2 * prob.n + prob.m + 1)
            for mode, kw in (("reverse", dict(lam=lam, obj_factor=obj)), ("forward", dict(v=v))):
                mkw = dict(lam=lam, obj=obj) if mode == "reverse" else dict(v=v)
                for _ in range(2):
                    fused = prob.JacobianProducts(x, **kw)
                    mat = mat_path(x, **mkw)
                    mat_path.index_add(x, **mkw)
                torch.cuda.synchronize()
                same = identical(fused, mat)
                t_f = time_ms(lambda: prob.JacobianProducts(x, **kw), a.reps)
                t_m = time_ms(lambda: mat_path(x, **mkw), a.reps)
                t_ia = time_ms(lambda: mat_path.index_add(x, **mkw), a.reps)
                gbs = bytes_inst * N / t_f / 1e6
                lines.append(f"{name:<15}{N:>9}{mode:>9}{bytes_inst:>8}{t_f:>10.3f}{gbs:>8.0f}{gbs / HBM_GBS:>8.1%}{t_m:>10.3f}"
                             f"{t_m / t_f:>10.2f}{t_ia:>14.3f}  {str(same).lower()}")
                print(lines[-1], flush=True)
                del fused, mat
            del x, lam, obj, v
            torch.cuda.empty_cache()
    text = "\n".join(lines) + "\n"
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
