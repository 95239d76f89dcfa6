"""torch.autograd face of c5_render_grad: the pre-cast image as a differentiable function of the cells' fields.

    from course5_b200 import api, autograd
    ctx = api.Context()
    ctx.upload_mesh(points, tets, alpha0, q0)          # topology and BVH, once
    alpha = torch.tensor(alpha0, requires_grad=True)   # float64, one value per tet: CPU, or CUDA on ctx's device
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

The fields' device picks the path. CPU tensors go through host memory as above. CUDA float64 tensors on
the context's device (single-device contexts) stay there: forward is c5_update_fields_device and
c5_render_device, backward c5_render_grad_device, all enqueued on torch.cuda.current_stream() with no host
synchronisation, so a whole fit step (forward, loss, backward, optimiser) runs on the device. On that path
a ray stopped by the step cap (C5_E_WALK, impossible on a valid mesh) is not reported.

light_curve(ctx, views, alpha, q) is the differentiable {sum tau, sum I} of each view (c5_render_flux
totals). On CUDA tensors its forward is the pipelined c5_render_flux_submit loop over the context's
views_in_flight lanes (one host wait per curve), and its backward is one c5_render_flux_grad_device call
over all views, on the same lanes, with grad_output read in place and no host synchronisation. On CPU
tensors it renders the views one by one and its backward is one c5_render_grad per view against g filled
with that view's upstream gradient.
"""
from __future__ import annotations

import numpy as np
import torch

from . import api, sweep


def _raw_view(view: api.View) -> api.View:
    v = api.View.from_buffer_copy(view)
    v.round_through_float = 0
    return v


def _band(view: api.View) -> tuple[int, int]:
    if view.row_begin == 0 and view.row_end == 0:
        return 0, view.res_y
    return view.row_begin, view.row_end


def _on_device(ctx: api.Context, alpha: torch.Tensor, q: torch.Tensor) -> bool:
    """True for CUDA fields, False for CPU ones; ValueError for anything else."""
    devices = {alpha.device.type, q.device.type}
    if devices == {"cpu"}:
        want = torch.device("cpu")
    elif devices == {"cuda"}:
        want = torch.device("cuda", ctx.devices[0])
    else:
        raise ValueError("alpha and q must both be CPU tensors or both CUDA tensors on the context's device")
    for name, t in (("alpha", alpha), ("q", q)):
        if t.dtype != torch.float64 or t.device != want or t.dim() != 1:
            raise ValueError(f"{name} must be a 1-D float64 tensor (one value per tet) on the CPU or on the "
                             f"context's device ({want})")
    return want.type == "cuda"


def _stream(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _fields(ctx: api.Context, alpha: torch.Tensor, q: torch.Tensor):
    if not _on_device(ctx, alpha, q):
        ctx.update_fields(alpha.detach().numpy(), q.detach().numpy())
        return ctx.fields_version
    n_tets = ctx.n_tets
    if n_tets and (alpha.shape[0] != n_tets or q.shape[0] != n_tets):
        raise ValueError("alpha and q need one value per tet of the uploaded mesh")
    a, b = alpha.detach().contiguous(), q.detach().contiguous()
    # stream-ordered: a and b, if they are copies, go back to torch's cache only for later work on this stream
    ctx.update_fields_device(a.data_ptr(), b.data_ptr(), _stream(alpha.device))
    return ctx.fields_version


class _Render(torch.autograd.Function):
    @staticmethod
    def forward(fn_ctx, ctx: api.Context, view: api.View, alpha: torch.Tensor, q: torch.Tensor):
        v = _raw_view(view)
        fn_ctx.version = _fields(ctx, alpha, q)
        fn_ctx.save_for_backward(alpha, q)
        fn_ctx.c5 = ctx
        fn_ctx.view = v
        if alpha.device.type == "cpu":
            return torch.from_numpy(ctx.render_raw(v).image)
        rb, re = _band(v)
        img = torch.zeros((v.res_y, v.res_x, 2), dtype=torch.float64, device=alpha.device)
        ctx.render_device(v, img[rb:re].data_ptr(), _stream(alpha.device), stats=False)
        return img

    @staticmethod
    def backward(fn_ctx, grad_output: torch.Tensor):
        ctx: api.Context = fn_ctx.c5
        alpha, q = fn_ctx.saved_tensors
        if ctx.fields_version != fn_ctx.version:  # another forward ran in between: put this one's fields back
            fn_ctx.version = _fields(ctx, alpha, q)
        want_alpha, want_q = fn_ctx.needs_input_grad[2], fn_ctx.needs_input_grad[3]
        if not (want_alpha or want_q):
            return None, None, None, None
        if alpha.device.type == "cpu":
            g = grad_output.detach().to(dtype=torch.float64, device="cpu").contiguous().numpy()
            ga, gq = ctx.render_grad(fn_ctx.view, g, alpha=want_alpha, q=want_q)
            return (None, None, torch.from_numpy(ga) if want_alpha else None,
                    torch.from_numpy(gq) if want_q else None)
        rb, re = _band(fn_ctx.view)
        g = grad_output.detach().to(dtype=torch.float64, device=alpha.device)[rb:re].contiguous()
        ga, gq = _grad_device(ctx, fn_ctx.view, g, alpha, want_alpha, want_q)
        return None, None, ga, gq


def _grad_device(ctx, view, g, alpha, want_alpha, want_q):
    """c5_render_grad_device of band-sized g into new CUDA tensors (None for one not wanted), enqueued only."""
    ga = torch.empty_like(alpha) if want_alpha else None
    gq = torch.empty_like(alpha) if want_q else None
    ctx.render_grad_device(view, g.data_ptr(), ga.data_ptr() if want_alpha else 0, gq.data_ptr() if want_q else 0,
                           stream=_stream(alpha.device), stats=False)
    return ga, gq


def render(ctx: api.Context, view: api.View, alpha: torch.Tensor, q: torch.Tensor) -> torch.Tensor:
    """The (res_y, res_x, 2) raw {tau, I} image of `view` for cell fields alpha and q (float64, one value per
    tet in the order given to upload_mesh; CPU, or CUDA on the context's device), differentiable in both.
    The image is on the fields' device; rows outside the view's band are 0."""
    return _Render.apply(ctx, view, alpha, q)


class _LightCurve(torch.autograd.Function):
    @staticmethod
    def forward(fn_ctx, ctx: api.Context, views, alpha: torch.Tensor, q: torch.Tensor):
        vs = [_raw_view(v) for v in views]
        fn_ctx.version = _fields(ctx, alpha, q)
        if alpha.device.type == "cuda":
            totals = sweep.render_light_curve(ctx, vs, in_flight=ctx.views_in_flight)[0][:, 0]
        else:
            totals = np.stack([ctx.render_flux(v)[1][0] for v in vs])  # (n_views, 2): {sum tau, sum I}
        fn_ctx.save_for_backward(alpha, q)
        fn_ctx.c5 = ctx
        fn_ctx.views = vs
        return torch.from_numpy(totals).to(alpha.device)

    @staticmethod
    def backward(fn_ctx, grad_output: torch.Tensor):
        ctx: api.Context = fn_ctx.c5
        alpha, q = fn_ctx.saved_tensors
        if ctx.fields_version != fn_ctx.version:
            fn_ctx.version = _fields(ctx, alpha, q)
        want_alpha, want_q = fn_ctx.needs_input_grad[2], fn_ctx.needs_input_grad[3]
        if not (want_alpha or want_q):
            return None, None, None, None
        if alpha.device.type == "cuda":
            # every view's {g_tau, g_I} read in place by the kernels: no fill, no host synchronisation
            go = grad_output.detach().to(dtype=torch.float64, device=alpha.device).contiguous()
            ga = torch.empty_like(alpha) if want_alpha else None
            gq = torch.empty_like(alpha) if want_q else None
            ctx.render_flux_grad_device(fn_ctx.views, go.data_ptr(), ga.data_ptr() if want_alpha else 0,
                                        gq.data_ptr() if want_q else 0, stream=_stream(alpha.device), stats=False)
            return None, None, ga, gq
        go = grad_output.detach().to(dtype=torch.float64, device="cpu")
        sums = [torch.zeros_like(alpha) if want_alpha else None, torch.zeros_like(alpha) if want_q else None]
        for k, v in enumerate(fn_ctx.views):
            # the flux is the image summed over the pixels outside the solid mask: its upstream gradient
            # is grad_output[k] in every pixel, and the gradient pass skips masked and background pixels
            rb, re = _band(v)
            g = np.zeros((v.res_y, v.res_x, 2))
            g[rb:re] = go[k].numpy()
            parts = [None if x is None else torch.from_numpy(x)
                     for x in ctx.render_grad(v, g, alpha=want_alpha, q=want_q)]
            for s, p in zip(sums, parts):
                if s is not None:
                    s += p
        return None, None, sums[0], sums[1]


def light_curve(ctx: api.Context, views, alpha: torch.Tensor, q: torch.Tensor) -> torch.Tensor:
    """(n_views, 2): the {sum tau, sum I} of each view over the pixels outside the solid mask (the totals of
    c5_render_flux, bit for bit, each view taken with round_through_float = 0) for cell fields alpha and q
    (as for render: float64, CPU or CUDA on the context's device), differentiable in both. Row bands are
    honoured. The cells' own fields only, not uploaded channels."""
    return _LightCurve.apply(ctx, list(views), alpha, q)
