"""torch.autograd face of c5_render_grad: the pre-cast image as a differentiable function of the cells' fields.

    from course5_b200 import api, autograd
    ctx = api.Context()
    ctx.upload_mesh(points, tets, alpha0, q0)          # topology and BVH, once
    alpha = torch.tensor(alpha0, requires_grad=True)   # CPU float64, one value per tet
    q = torch.tensor(q0, requires_grad=True)
    img = autograd.render(ctx, view, alpha, q)          # (res_y, res_x, 2): {tau, I}
    loss = ((img[..., 1] - observed) ** 2)[mask].sum()
    loss.backward()                                     # alpha.grad, q.grad

Forward uploads the fields (c5_update_fields: no topology or BVH rebuild) and renders the raw image
(c5_render_raw with round_through_float = 0: the float cast has no useful derivative). Backward is one
c5_render_grad against grad_output. If the context's fields changed between the two (another forward, or
an update_fields call), backward first uploads again the fields its forward saw. Pixels under the solid
mask are NaN in the image; exclude them from the loss (they add nothing to the gradients). Gradients are
summed with FP64 atomics on the device: equal to rounding, not bit for bit, from run to run.
"""
from __future__ import annotations

import torch

from . import api


def _raw_view(view: api.View) -> api.View:
    v = api.View.from_buffer_copy(view)
    v.round_through_float = 0
    return v


def _fields(ctx: api.Context, alpha: torch.Tensor, q: torch.Tensor):
    for name, t in (("alpha", alpha), ("q", q)):
        if t.dtype != torch.float64 or t.device.type != "cpu" or t.dim() != 1:
            raise ValueError(f"{name} must be a 1-D CPU float64 tensor (one value per tet)")
    ctx.update_fields(alpha.detach().numpy(), q.detach().numpy())
    return ctx.fields_version


class _Render(torch.autograd.Function):
    @staticmethod
    def forward(fn_ctx, ctx: api.Context, view: api.View, alpha: torch.Tensor, q: torch.Tensor):
        v = _raw_view(view)
        fn_ctx.version = _fields(ctx, alpha, q)
        img = ctx.render_raw(v).image
        fn_ctx.save_for_backward(alpha, q)
        fn_ctx.c5 = ctx
        fn_ctx.view = v
        return torch.from_numpy(img)

    @staticmethod
    def backward(fn_ctx, grad_output: torch.Tensor):
        ctx: api.Context = fn_ctx.c5
        alpha, q = fn_ctx.saved_tensors
        if ctx.fields_version != fn_ctx.version:  # another forward ran in between: put this one's fields back
            fn_ctx.version = _fields(ctx, alpha, q)
        want_alpha, want_q = fn_ctx.needs_input_grad[2], fn_ctx.needs_input_grad[3]
        if not (want_alpha or want_q):
            return None, None, None, None
        g = grad_output.detach().to(dtype=torch.float64, device="cpu").contiguous().numpy()
        ga, gq = ctx.render_grad(fn_ctx.view, g, alpha=want_alpha, q=want_q)
        return (None, None, torch.from_numpy(ga) if want_alpha else None,
                torch.from_numpy(gq) if want_q else None)


def render(ctx: api.Context, view: api.View, alpha: torch.Tensor, q: torch.Tensor) -> torch.Tensor:
    """The (res_y, res_x, 2) raw {tau, I} image of `view` for cell fields alpha and q (CPU float64, one
    value per tet in the order given to upload_mesh), differentiable in both."""
    return _Render.apply(ctx, view, alpha, q)

