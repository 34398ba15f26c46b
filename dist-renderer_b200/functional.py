"""decode_sdf / decode_sdf_gradient -- drop-ins for core/utils/decoder_utils.py:53-92 on the CUDA engines."""
import torch

from . import _abi
from .plan import plan_for

_ENGINES = {"simt": _abi.ENGINE_SIMT, "tc": _abi.ENGINE_TC}
DEFAULT_ENGINE = "auto"


def resolve_engine(plan, engine):
    """'auto' picks the tensor-core engine when the network shape is covered by it, else the fp32 SIMT engine."""
    if engine in (None, "auto"):
        from . import tc
        return _abi.ENGINE_TC if tc.supported(plan) else _abi.ENGINE_SIMT
    if engine == "tc":
        from . import tc
        if not tc.supported(plan):
            raise NotImplementedError("the tensor-core engine does not cover this decoder shape / device")
        return _abi.ENGINE_TC
    return _ENGINES[engine]


def _stream(device):
    """The caller's current stream on `device` (the tensors' device, not whatever device is current)."""
    return torch.cuda.current_stream(device).cuda_stream


def _check_device(plan, points):
    if points.device != plan.device:
        raise ValueError("points live on %s but the decoder on %s" % (points.device, plan.device))


def _check_points(points):
    if points.dim() != 2 or points.shape[1] != 3:
        raise ValueError("points must be (K, 3)")
    if not points.is_cuda:
        raise ValueError("points must be a CUDA tensor (no CPU path)")


class _DecodeFn(torch.autograd.Function):
    """Decoder rows on the CUDA engines, (K, n_out).  The kernels compute one output per launch: a multi-output network
    (the colour decoder) is evaluated output by output, every hidden layer shared (plan.c_net(out_index=...))."""

    @staticmethod
    def forward(ctx, latent, points, plan, clamp_dist, engine, index=None):
        lib = _abi.lib()
        _check_device(plan, points)
        # index (int32, one entry per row) picks each row's code among the C rows of `latent` (dist_net_t.row_code)
        n_codes = latent.shape[0] if index is not None else 1
        with torch.cuda.device(plan.device):
            st = _stream(plan.device)
            pts = points.detach().float().contiguous()
            n = pts.shape[0]
            cols = []
            cd = float(clamp_dist) if clamp_dist is not None else 0.0
            for c in range(plan.n_out):
                net, engine, _keep = plan.net_for(latent, engine, st, out_index=c, n_codes=n_codes)
                if n_codes > 1:
                    net.row_code = index.data_ptr()
                out = torch.empty(n, device=pts.device, dtype=torch.float32)
                if n > 0:
                    _abi.check(lib.dist_decoder_forward(net, engine, _abi.ptr(pts), n, None, cd, _abi.ptr(out), st))
                cols.append(out)
            sdf = torch.stack(cols, 1) if plan.n_out > 1 else cols[0].reshape(n, 1)
        ctx.plan, ctx.cd, ctx.engine, ctx.n_codes = plan, cd, engine, n_codes
        ctx.save_for_backward(pts, latent if latent is not None else torch.empty(0, device=pts.device),
                              index if n_codes > 1 else torch.empty(0, device=pts.device))
        ctx.has_latent = latent is not None
        return sdf

    @staticmethod
    def backward(ctx, g):
        pts, latent, index = ctx.saved_tensors
        plan, lib, n_codes = ctx.plan, _abi.lib(), ctx.n_codes
        with torch.cuda.device(plan.device):
            st = _stream(plan.device)
            n = pts.shape[0]
            dpts = torch.zeros(n, 3, device=pts.device)
            acc0, accl = plan.acc_buffers(n_codes)
            gd = g.detach().float()
            for c in range(plan.n_out):
                net, eng_b, _keep = plan.net_for(latent if ctx.has_latent else None, ctx.engine, st, out_index=c,
                                                 n_codes=n_codes)
                if n_codes > 1:
                    net.row_code = index.data_ptr()
                coef = gd[:, c].contiguous()
                dp = torch.empty(n, 3, device=pts.device)
                if n > 0:
                    _abi.check(lib.dist_decoder_backward(net, eng_b, _abi.ptr(pts), _abi.ptr(coef), None, n, None, ctx.cd,
                                                         _abi.ptr(dp), _abi.ptr(acc0), _abi.ptr(accl), st))
                    dpts += dp
        g_lat = plan.latent_grad(acc0, accl, n_codes).reshape(latent.shape) \
            if (ctx.has_latent and ctx.needs_input_grad[0]) else None
        return g_lat, (dpts if ctx.needs_input_grad[1] else None), None, None, None, None


def _check_index(latent, latent_index, points):
    """(C, L) codes + one int index per row in [0, C) -> the int32 row-code array of the kernels."""
    if not torch.is_tensor(latent) or latent.dim() != 2:
        raise ValueError("latent_index needs latent of shape (C, L)")
    if not torch.is_tensor(latent_index) or latent_index.dim() != 1 or latent_index.shape[0] != points.shape[0]:
        raise ValueError("latent_index must be a 1-D tensor with one entry per point (%d)" % points.shape[0])
    if latent_index.dtype.is_floating_point or latent_index.dtype.is_complex or latent_index.dtype == torch.bool:
        raise ValueError("latent_index must be an integer tensor")
    C = latent.shape[0]
    if latent_index.numel() and (int(latent_index.min()) < 0 or int(latent_index.max()) >= C):
        raise ValueError("latent_index values must be in [0, %d)" % C)
    return latent_index.to(device=points.device, dtype=torch.int32).contiguous()


def decode_sdf(decoder, latent_vector, points, clamp_dist=0.1, MAX_POINTS=100000, no_grad=False, engine=None,
               latent_index=None):
    """sdf (K,1) of `points` (K,3) for one latent code (1,L).  decoder_utils.py:53-74.

    MAX_POINTS is accepted for signature compatibility; the fused engines tile rows internally (64-128 rows per
    CTA resident in shared memory) so no host-side chunking is needed.  Differentiable w.r.t. latent and points.

    latent_index (extension, no counterpart in the reference): with `latent_vector` of shape (C, L) and an integer
    tensor (K,) of values in [0, C), row i is decoded with code latent_index[i] -- bit for bit what
    decode_sdf(decoder, latent_vector[c:c+1], points[i:i+1]) gives on the same engine -- in one launch; the gradient
    reaches all C codes, (C, L).
    """
    _check_points(points)
    plan = plan_for(decoder)
    if plan.n_out != 1:
        raise ValueError("decode_sdf expects a single-output decoder (use decode_color for the colour network)")
    index = _check_index(latent_vector, latent_index, points) if latent_index is not None else None
    eng = resolve_engine(plan, engine or DEFAULT_ENGINE)
    if no_grad:
        with torch.no_grad():
            return _DecodeFn.apply(latent_vector, points, plan, clamp_dist, eng, index)
    return _DecodeFn.apply(latent_vector, points, plan, clamp_dist, eng, index)


def decode_sdf_gradient(decoder, latent_vector, points, clamp_dist=0.1, MAX_POINTS=100000, no_grad=False,
                        engine=None):
    """d clamp(sdf)/d xyz (K,3) by the fused forward + transposed chain.  decoder_utils.py:76-92.

    The reference builds this with autograd (create_graph=True); for ReLU / weight-norm decoders the result is
    piecewise constant in (xyz, latent), so its own derivative is zero almost everywhere and the returned tensor
    carries no graph.  The reference's grad_outputs quirk (ones shaped like the points, i.e. an implied factor 3
    on torch 1.1 -- SURVEY.md H7) is not reproduced: this is the plain gradient.
    """
    _check_points(points)
    lib = _abi.lib()
    plan = plan_for(decoder)
    eng = resolve_engine(plan, engine or DEFAULT_ENGINE)
    _check_device(plan, points)
    with torch.cuda.device(plan.device):
        st = _stream(plan.device)
        net, eng, _keep = plan.net_for(latent_vector, eng, st)
        pts = points.detach().float().contiguous()
        n = pts.shape[0]
        grad = torch.empty(n, 3, device=pts.device)
        cd = float(clamp_dist) if clamp_dist is not None else 0.0
        if n > 0:
            _abi.check(lib.dist_decoder_input_grad(net, eng, _abi.ptr(pts), n, None, cd, _abi.ptr(grad), None, st))
    return grad


def decode_color(decoder, color_code, shape_code, points, MAX_POINTS=100000, no_grad=False, engine=None):
    """rgb (K,3) of `points` (K,3) from a colour decoder fed [shape code | colour code | xyz] rows --
    decoder_utils.py:94-112 (used by SDFRenderer_color, renderer_rgb.py:33).

    The colour network (``last_dim = 3``, latent = shape code + colour code) runs on the same fused engines as the SDF
    network: both codes are folded into the per-render biases, the hidden layers run on tcgen05 (or exact fp32), and the
    three outputs are three dot-product epilogues over the shared hidden layers (three launches of the single-output
    kernel; a render queries the colour network once per hit pixel, ~1e-3 of its decoder rows).  Differentiable w.r.t.
    both codes and the points.  MAX_POINTS is accepted for signature compatibility (no host-side chunking needed)."""
    _check_points(points)
    plan = plan_for(decoder)
    if plan.n_out != 3:
        raise ValueError("decode_color expects a decoder with three outputs (last_dim=3)")
    eng = resolve_engine(plan, engine or DEFAULT_ENGINE)
    latent = torch.cat([shape_code.reshape(1, -1), color_code.reshape(1, -1)], 1)      # decoder_utils.py:103
    if no_grad:
        with torch.no_grad():
            return _DecodeFn.apply(latent, points, plan, None, eng)
    return _DecodeFn.apply(latent, points, plan, None, eng)
