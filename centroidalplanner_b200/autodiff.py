"""The batched constraints and cost as a differentiable torch function.

`constraints_and_cost(problem, x)` returns g (N, m) and the cost (N,) of `problem.eval` at x (N, n), and lets gradients flow back to
x: in reverse mode the backward pass is ONE fused product x_bar = grad_cost * grad f(x) + J(x)^T grad_g, in forward mode the tangent
is ONE fused product (J(x) v, grad f(x) . v) -- cplb_jacobian_products_device in both cases, so the Jacobian is never materialised.
Only x is differentiable: derivatives with respect to the per-instance parameters and second derivatives are not provided.
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable


def _plain(t):
    """The tensor that holds t's memory: torch.func transforms hand a Function's rules wrapper tensors without storage, and the
    library reads raw device pointers."""
    while torch._C._functorch.is_functorch_wrapped_tensor(t):
        t = torch._C._functorch.get_unwrapped(t)
    return t


class _ConstraintsAndCost(torch.autograd.Function):
    @staticmethod
    def forward(x, problem, per_instance):
        out = problem.eval(x, g=True, jac=False, cost=True, per_instance=per_instance)
        return out["g"], out["cost"]

    @staticmethod
    def setup_context(ctx, inputs, output):
        x, problem, per_instance = inputs
        ctx.problem, ctx.per_instance = problem, per_instance
        ctx.save_for_backward(x)
        ctx.save_for_forward(x)
        ctx.set_materialize_grads(False)  # an unused output hands back None, which the product takes as NULL

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_g, grad_cost):
        if grad_g is None and grad_cost is None:
            return None, None, None
        (x,) = ctx.saved_tensors
        lam = None if grad_g is None else grad_g.contiguous()
        of = None if grad_cost is None else grad_cost.contiguous()
        return ctx.problem.JacobianProducts(x, lam=lam, obj_factor=of, per_instance=ctx.per_instance)["x_bar"], None, None

    @staticmethod
    def jvp(ctx, x_dot, _problem_dot, _per_instance_dot):
        if x_dot is None:
            return None, None
        (x,) = ctx.saved_tensors
        with torch._C._DisableFuncTorch():  # the outputs are allocated as plain tensors too
            out = ctx.problem.JacobianProducts(_plain(x), v=_plain(x_dot).contiguous(), per_instance=ctx.per_instance)
        return out["g_dot"], out["f_dot"]


def constraints_and_cost(problem, x, per_instance=None):
    """g (N, m) and cost (N,) of `problem` (a BatchedCplProblem) at x, a float64 CUDA tensor (N, n), differentiable in x.

    Reverse mode (`backward`, `torch.autograd.grad`) runs one fused reverse product, with grad_g as the multipliers and grad_cost as
    the objective factor; forward mode (`torch.func.jvp`, `torch.autograd.forward_ad`) one fused forward product.  The backward
    pass cannot itself be differentiated (a double backward raises).  per_instance: dict of per-instance parameter arrays as for
    `problem.eval`; they enter as constants, so none of them may require grad."""
    for name, t in (per_instance or {}).items():
        if torch.is_tensor(t) and t.requires_grad:
            raise ValueError(f"per-instance array '{name}' requires grad: derivatives with respect to the parameters are not provided")
    return _ConstraintsAndCost.apply(x.contiguous(), problem, per_instance)
