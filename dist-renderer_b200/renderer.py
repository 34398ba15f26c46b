"""SDFRenderer -- drop-in for core/sdfrenderer/renderer.py:12-999 on the B200 engines.

Same constructor and method signatures as the reference class; ``render_depth`` / ``render_normal`` / ``render``
return tensors with the reference's shapes, dtypes and autograd connectivity (to ``latent``, ``R``, ``T`` according
to the ``no_grad_*`` flags).  Everything per-ray runs in libdist_b200.so; PyTorch here only allocates buffers,
launches on the current stream and chains the tiny camera Jacobian (c = -R^T T, ray = normalize(R^T K^-1 u)).

Differences from the reference, all loud:
  * no CPU path: ``use_gpu=False`` or a CPU decoder raises;
  * ``sample_index_type != 'min_abs'`` raises NotImplementedError (no caller in the reference uses another type);
    ``pyramid_recursive`` is implemented for the default ``scale_list=[4,2,1]`` on full images;
  * 3x4 ``transform_matrix`` raises (the reference's own 3x4 inverse path calls an un-imported ``pdb``);
  * when no ray meets the unit sphere the reference dies inside ``.max()`` of an empty tensor; here
    ``ValueError('No valid depth.')`` (renderer.py:215) is raised;
  * new: ``render_silhouette`` = the (mask, min_abs_query) pair; ``rows=(row0, row_step, n_rows)`` renders a band
    of image rows for ray-tile sharding across GPUs (parallel.py); ``render_views`` marches V poses of one shape in
    one fused call.
"""
import os

import numpy as np
import torch

from . import _abi
from .functional import resolve_engine, DEFAULT_ENGINE
from .plan import plan_for

_MARCH = {"trivial": _abi.MARCH_TRIVIAL, "trivial_non_parallel": _abi.MARCH_TRIVIAL,
          "recursive": _abi.MARCH_RECURSIVE, "pyramid_recursive": _abi.MARCH_PYRAMID}


def _stream(device=None):
    """The caller's current stream ON THE RENDERER'S DEVICE (not on whatever device happens to be current)."""
    return torch.cuda.current_stream(device).cuda_stream


class _RenderDepthFn(torch.autograd.Function):
    """Forward: dist_render_depth_fwd.  Backward: dist_render_depth_bwd + host camera chain (SURVEY.md H6)."""

    @staticmethod
    def forward(ctx, latent, R, T, ren, opts):
        with torch.cuda.device(ren.device):     # the library launches on the current device: make it the renderer's
            return _RenderDepthFn._forward(ctx, latent, R, T, ren, opts)

    @staticmethod
    def _forward(ctx, latent, R, T, ren, opts):
        lib, st = _abi.lib(), _stream(ren.device)
        plan = ren.plan
        plan.refresh()
        dev = ren.device
        P, B = ren.P, ren.buffer_size
        engine = resolve_engine(plan, opts["engine"])
        n_codes = ren._n_codes(latent)     # > 1: view v is rendered with latent[v]
        net, engine, _keep = plan.net_for(latent, engine, st, n_codes=n_codes)
        Rd = R.detach().float().contiguous()
        if Rd.shape != ((3, 3) if ren.n_views == 1 and R.dim() == 2 else (ren.n_views, 3, 3)):
            raise ValueError("R must be (3,3), or (n_views,3,3) on a multi-view renderer")
        cam_pos = ren.get_camera_location(Rd, T.detach().float()).contiguous()  # renderer.py:186
        cam = ren._c_camera(Rd, cam_pos, opts["use_transform"])
        mp = _abi.March(ren.march_step, B, _MARCH[opts["kind"]], 1 if opts["kind"] != "pyramid_recursive" else 0,
                        ren.ray_marching_ratio, ren.threshold, float(opts["clamp_dist"]), opts["replay"])
        pyr = opts["kind"] == "pyramid_recursive"
        if pyr:
            mp.coarse_steps[0], mp.coarse_steps[1] = ren._coarse_steps()
        mp.cam_grad_levels = opts["cam_levels"]
        # two-tier precision of the march rows (tc.py): only on the tensor-core engine, only when the one-pass values of
        # this decoder were measured to be accurate to half the margin
        screen = plan.tc.get("screen") if (engine == _abi.ENGINE_TC and plan.tc is not None and ren.screen) else None
        if screen:
            mp.screen, mp.screen_margin = 1, screen["margin"]
            mp.screen_tpred, mp.screen_ext_margin = ren.screen_tpred, ren.screen_ext_margin
        f32 = dict(device=dev, dtype=torch.float32)
        saved = {
            "flags": torch.empty(P, device=dev, dtype=torch.uint8), "nreal": torch.empty(P, device=dev, dtype=torch.int32),
            "top_sdf": torch.empty(B, P, **f32), "top_pt": torch.empty(B, 3, P, **f32),
            "top_zafter": torch.empty(B, P, **f32), "top_zgen": torch.empty(B, P, **f32),
            # sdf at the origin: one per view (the views' own codes when each view has one)
            "sdf_origin": torch.empty(ren.n_views, **f32), "dist": torch.empty(P, **f32),
            "top_lvl": torch.empty(B, P, device=dev, dtype=torch.uint8),
        }
        scr = ren._scratch(pyramid=pyr)
        # ReLU-mask cache (dist_workspace_t.mask_buf): when a backward will follow, the forward keeps the sign bits of the rows
        # it evaluates at full precision (512 B per row for the 8x512 network), so that the backward replays the transposed
        # chain alone.  Sized for `mask_rows_per_ray` such rows per ray; rows beyond that fall back to the full replay.
        mask_cap = 0
        if screen and ren.mask_cache and (opts["want_depth_grad"] or opts["want_mask_grad"]):
            mask_cap = (int(ren.mask_rows_per_ray * P) + 127) // 128 * 128
            saved["mask_buf"] = torch.empty(16 * (plan.n_layers - 1) * mask_cap, device=dev, dtype=torch.int32)
            saved["top_slot"] = torch.empty(B, P, device=dev, dtype=torch.int32)
        ws = _abi.Workspace()
        for name in _abi.WS_FIELDS:
            if name == "mask_cap":
                continue
            t = saved.get(name, scr.get(name))
            setattr(ws, name, t.data_ptr() if t is not None else None)
        ws.mask_cap = mask_cap
        ws.tile_counters = ren.tile_counters.data_ptr()
        Zdepth = torch.empty(P, **f32)
        mask = torch.empty(P, device=dev, dtype=torch.uint8)
        min_sdf = torch.empty(P, **f32)
        _abi.check(lib.dist_render_depth_fwd(net, engine, cam, mp, ws, _abi.ptr(Zdepth), _abi.ptr(mask),
                                             _abi.ptr(min_sdf), _abi.ptr(ren.rows_evaluated), st))
        ren._last_counts = scr["view_stat"]
        ctx.ren, ctx.opts, ctx.engine, ctx.mp, ctx.mask_cap, ctx.n_codes = ren, opts, engine, mp, mask_cap, n_codes
        ctx.saved = saved
        ctx.save_for_backward(latent, Rd, T.detach().float())
        hit = saved["flags"].bitwise_and(1).bool()
        ctx.mark_non_differentiable(mask, hit)
        # NB: nothing stored on ctx may also be returned (tensor -> grad_fn -> ctx -> tensor would be a reference cycle
        # that only the cyclic GC frees, i.e. ~60 MB of saved samples per render lingering for many steps)
        return Zdepth, mask, min_sdf, hit

    @staticmethod
    def backward(ctx, gZ, _gmask, gM, _ghit):
        with torch.cuda.device(ctx.ren.device):
            return _RenderDepthFn._backward(ctx, gZ, gM)

    @staticmethod
    def _backward(ctx, gZ, gM):
        latent, Rd, Td = ctx.saved_tensors
        ren, opts, lib, st = ctx.ren, ctx.opts, _abi.lib(), _stream(ctx.ren.device)
        plan, dev, P, B = ren.plan, ren.device, ren.P, ren.buffer_size
        net, eng_b, _keep = plan.net_for(latent, ctx.engine, st, n_codes=ctx.n_codes)
        cam_pos = ren.get_camera_location(Rd, Td).contiguous()
        cam = ren._c_camera(Rd, cam_pos, opts["use_transform"])
        V, Pv = ren.n_views, ren.Pv
        scr = ren._scratch()
        ws = _abi.Workspace()
        for name in _abi.WS_FIELDS:
            if name == "mask_cap":
                continue
            t = ctx.saved.get(name, scr.get(name))
            setattr(ws, name, t.data_ptr() if t is not None else None)
        ws.mask_cap = ctx.mask_cap
        pyr = opts["kind"] == "pyramid_recursive"
        gZ = gZ.contiguous().float() if (gZ is not None and opts["want_depth_grad"]) else None
        gM = gM.contiguous().float() if (gM is not None and opts["want_mask_grad"]) else None
        want_cam = opts["cam_levels"] != 0 and (ctx.needs_input_grad[1] or ctx.needs_input_grad[2])
        f32 = dict(device=dev, dtype=torch.float32)
        acc0, accl = plan.acc_buffers(ctx.n_codes)
        d_cam = torch.zeros(V, 3, **f32) if want_cam else None
        d_ray = torch.zeros(3, P, **f32) if want_cam else None
        n_coarse = V * sum(g[0].shape[1] for g in ren._coarse_homo()) if (want_cam and pyr) else 0
        d_ray_c = torch.zeros(3 * n_coarse, **f32) if n_coarse else None
        g_lat = g_R = g_T = None
        if gZ is not None or gM is not None:
            s_row, s_pts, s_coef, s_dpts, s_cnt = scr["b_row"], scr["b_pts"], scr["b_coef"], scr["b_dpts"], scr["b_cnt"]
            _abi.check(lib.dist_render_depth_bwd(net, eng_b, cam, ctx.mp, ws, _abi.ptr(gZ), _abi.ptr(gM),
                                                 _abi.ptr(acc0), _abi.ptr(accl), _abi.ptr(d_cam), _abi.ptr(d_ray),
                                                 _abi.ptr(d_ray_c), _abi.ptr(s_row), _abi.ptr(s_pts), _abi.ptr(s_coef), None,
                                                 _abi.ptr(s_dpts), _abi.ptr(s_cnt), _abi.ptr(ren.rows_grad), st))
            if ctx.needs_input_grad[0] and latent is not None:
                g_lat = plan.latent_grad(acc0, accl, ctx.n_codes).reshape(latent.shape).to(latent.dtype)
            if want_cam:
                with torch.enable_grad():
                    Rg, Tg = Rd.clone().requires_grad_(True), Td.clone().requires_grad_(True)
                    c = ren.get_camera_location(Rg, Tg)

                    def per_view(g, n):   # kernel layout [3][V*n] -> layout of the host tensor, (3,n) or (V,3,n)
                        return g.reshape(3, n) if Rg.dim() == 2 else g.reshape(3, V, n).permute(1, 0, 2)
                    outs, gouts = [c, ren.get_camera_rays(Rg)], [d_cam.reshape(c.shape), per_view(d_ray, Pv)]
                    if d_ray_c is not None:   # samples taken on the 1/2- and 1/4-resolution parent rays
                        off = 0
                        for (homo,) in ren._coarse_homo():
                            n_l = homo.shape[1]
                            outs.append(ren.get_camera_rays(Rg, homo=homo))
                            gouts.append(per_view(d_ray_c[off:off + 3 * V * n_l], n_l))
                            off += 3 * V * n_l
                    g_R, g_T = torch.autograd.grad(outs, [Rg, Tg], gouts, allow_unused=True)
        return g_lat, g_R, g_T, None, None


class SDFRenderer(object):
    def __init__(self, decoder, intrinsic, img_hw=None, transform_matrix=None, march_step=50, buffer_size=5,
                 ray_marching_ratio=1.5, use_depth2normal=False, max_sample_dist=0.2, radius=1.0, threshold=5e-5,
                 scale_list=[4, 2, 1], march_step_list=[3, 3, -1], use_gpu=True, is_eval=True, engine=None,
                 rows=None, screen=None, screen_tpred=0.30, screen_ext_margin=0.04, mask_cache=None, mask_rows_per_ray=9.0):
        # renderer.py:13-59
        self.decoder = decoder
        if use_gpu and torch.cuda.device_count() == 0:
            raise ValueError('No GPU device found.')  # renderer.py:51-52
        if not use_gpu:
            raise RuntimeError("dist-renderer_b200 has no CPU path: use_gpu=False is not supported")
        p = next(self.decoder.parameters())
        if not p.is_cuda:
            raise ValueError("the decoder must be on a CUDA device (no CPU path)")
        self.device = p.device
        if is_eval:
            self.decoder.eval()
        if not (1 <= buffer_size <= _abi.MAX_BUFFER):
            raise NotImplementedError("buffer_size must be in [1, %d]" % _abi.MAX_BUFFER)
        self.march_step, self.buffer_size = int(march_step), int(buffer_size)
        self.max_sample_dist = max_sample_dist
        self.ray_marching_ratio = float(ray_marching_ratio)
        self.use_depth2normal = use_depth2normal
        self.radius, self.threshold = float(radius), float(threshold)
        self.scale_list, self.march_step_list = scale_list, march_step_list
        self.engine = engine or DEFAULT_ENGINE
        if type(intrinsic) == torch.Tensor:
            intrinsic = intrinsic.detach().cpu().numpy()
        self.intrinsic = np.asarray(intrinsic, dtype=np.float64)
        if img_hw is None:
            img_hw = (int(self.intrinsic[1, 2] * 2), int(self.intrinsic[0, 2] * 2))
        self.img_hw = (int(img_hw[0]), int(img_hw[1]))
        h, w = self.img_hw
        # rows = (row0, row_step, n_rows[, row_group]): local row l is image row row0 + (l // g) * row_step + l % g
        self.rows = (0, 1, h, 1) if rows is None else (tuple(int(v) for v in rows) + (1,))[:4]
        row0, step, n_rows, grp = self.rows
        if not (0 <= row0 and step >= 1 and n_rows >= 1 and grp >= 1 and
                row0 + ((n_rows - 1) // grp) * step + (n_rows - 1) % grp < h):
            raise ValueError("rows=(row0,row_step,n_rows[,row_group]) outside the image")
        self.full_image = (row0 == 0 and step == grp and n_rows == h)
        self.local_hw = (n_rows, w)
        self.n_views = 1             # > 1 only on the children made by _fused_child (multi-view march, render_views)
        self.Pv = n_rows * w         # pixels per view
        self.P = self.Pv             # pixels per call = n_views * Pv
        self.K = torch.from_numpy(self.intrinsic).float().to(self.device)
        self.K_inv = torch.from_numpy(np.linalg.inv(self.intrinsic)).float().to(self.device)
        if transform_matrix is None:
            transform_matrix = np.array([[1., 0., 0.], [0., 0., -1.], [0., 1., 0.]])
        transform_matrix = np.asarray(transform_matrix, dtype=np.float64)
        if transform_matrix.shape != (3, 3):
            raise NotImplementedError("only 3x3 transform_matrix is supported (renderer.py:116 is dead code upstream)")
        self.transform_matrix = torch.from_numpy(transform_matrix).float().to(self.device)
        self.plan = plan_for(decoder)
        # decoder-row counters for roofline accounting: forward rows cost F flop, gradient rows (normal / backward
        # replay: forward + transposed chain) cost 2F
        self.rows_evaluated = torch.zeros(1, device=self.device, dtype=torch.int64)
        # [0] gradient rows evaluated as forward + transposed chain (2F: normals, full backward replay),
        # [1] backward rows replayed from the mask cache (transposed chain only, F)
        self.rows_grad = torch.zeros(2, device=self.device, dtype=torch.int64)
        # 128-row tile programs of the forward launches evaluated with [one fp16 pass, three split-precision passes]
        self.tile_counters = torch.zeros(2, device=self.device, dtype=torch.int64)
        # two-tier precision of the march (dist_march_t.screen): on unless switched off here or by DIST_SCREEN=0
        self.screen = (os.environ.get("DIST_SCREEN", "1") != "0") if screen is None else bool(screen)
        self.screen_tpred = float(os.environ.get("DIST_SCREEN_TPRED", screen_tpred))
        self.screen_ext_margin = float(os.environ.get("DIST_SCREEN_EXT", screen_ext_margin))
        # ReLU-mask cache for the backward (dist_workspace_t.mask_buf): on with the two precision tiers unless switched off
        self.mask_cache = (os.environ.get("DIST_MASK_CACHE", "1") != "0") if mask_cache is None else bool(mask_cache)
        self.mask_rows_per_ray = float(mask_rows_per_ray)
        self._homo_calib = None
        self._calib_map = None
        self._scr = None
        self._last_counts = None

    # ---- accessors of the reference ------------------------------------------------------------------------
    def get_intrinsic(self):
        return self.intrinsic

    def get_threshold(self):
        return self.threshold

    def get_img_hw(self):
        return self.img_hw

    @property
    def homo_calib(self):
        """K^-1 [x, y, 1] for the rendered rows, (3, P).  renderer.py:37-39."""
        if self._homo_calib is None:
            w = self.img_hw[1]
            ys = self._image_rows(torch.arange(self.rows[2], device=self.device)).float()
            xs = torch.arange(w, device=self.device).float()
            Y, X = torch.meshgrid(ys, xs, indexing="ij")
            homo = torch.stack([X.reshape(-1), Y.reshape(-1), torch.ones(self.Pv, device=self.device)], 0)
            self._homo_calib = torch.matmul(self.K_inv, homo)
        return self._homo_calib

    @property
    def calib_map(self):
        if self._calib_map is None:
            self._calib_map = self.normalize_vectors(self.homo_calib)[2, :]  # renderer.py:59
        return self._calib_map

    # The camera helpers accept one pose (R (3,3), T (3,)) -> (3,), (3,P) as in the reference, or a stack of poses
    # (R (V,3,3), T (V,3)) -> (V,3), (V,3,P).  A stack is evaluated pose by pose with the single-pose ops, so that a
    # fused multi-view render sees bit-identical cameras to V separate renders (batched GEMMs may round differently).
    def normalize_vectors(self, x):  # renderer.py:171-178
        return x.div(torch.norm(x, p=2, dim=0).expand_as(x) + 1e-12)

    def get_camera_location(self, R, T):  # renderer.py:180-188
        if R.dim() == 3:
            return torch.stack([self.get_camera_location(R[v], T[v]) for v in range(R.shape[0])], 0)
        return torch.matmul(-R.transpose(1, 0), T[:, None]).squeeze(1)

    def get_camera_rays(self, R, homo=None):  # renderer.py:190-200
        if R.dim() == 3:
            return torch.stack([self.get_camera_rays(R[v], homo) for v in range(R.shape[0])], 0)
        return self.normalize_vectors(torch.matmul(R.transpose(1, 0), self.homo_calib if homo is None else homo))

    def transform_points(self, points):  # renderer.py:84-98
        return torch.matmul(self.transform_matrix, points)

    def inv_transform_points(self, points):  # renderer.py:100-120
        return torch.matmul(self.transform_matrix.transpose(1, 0), points)

    def generate_point_samples(self, cam_pos, cam_rays, Zdepth, inv_transform=True, has_zdepth_grad=False):
        # renderer.py:202-223 (host-side helper kept for subclasses; the march generates its points in-kernel)
        if not has_zdepth_grad:
            Zdepth = Zdepth.detach()
        if Zdepth.shape[0] == 0:
            raise ValueError('No valid depth.')
        points = cam_rays * Zdepth[None, :] + cam_pos[:, None]
        if inv_transform:
            points = self.inv_transform_points(points)
        if not points.requires_grad:
            points.requires_grad = True
        return points

    def get_distance_from_origin(self, cam_pos, cam_rays):  # renderer.py:225-239
        if cam_rays.dim() == 3:
            return torch.stack([self.get_distance_from_origin(cam_pos[v], cam_rays[v]) for v in range(cam_rays.shape[0])], 0)
        ptq = (cam_pos[:, None] * cam_rays).sum(0)
        return torch.norm(cam_pos[:, None] - ptq[None, :] * cam_rays, p=2, dim=0)

    # ---- internals ------------------------------------------------------------------------------------------
    def _image_rows(self, local_rows):
        """Image row of each local row of this renderer's band (interleaved groups of `row_group` rows)."""
        row0, step, _, grp = self.rows
        return row0 + (local_rows // grp) * step + local_rows % grp

    def _transform_host(self):
        """Host copy of `transform_matrix` (9 floats for the camera descriptor).  Cached: reading the device tensor back on
        every call would make each render_depth / render_normal / backward wait for all queued GPU work.  The cache is keyed
        on the tensor object and its version counter, so assigning or modifying `self.transform_matrix` refreshes it."""
        tm = self.transform_matrix
        key = (id(tm), tm._version)
        if getattr(self, "_tm_host_key", None) != key:
            self._tm_host = tm.detach().cpu().numpy().astype(np.float32).reshape(-1)
            self._tm_host_key = key
        return self._tm_host

    def _c_camera(self, R, cam_pos, use_transform=True):
        cam = _abi.Camera()
        Kinv = np.linalg.inv(self.intrinsic).astype(np.float32).reshape(-1)
        Mn = self._transform_host()
        M = Mn if use_transform else np.eye(3).reshape(-1)
        for i in range(9):
            cam.Kinv[i], cam.M[i], cam.Mn[i] = float(Kinv[i]), float(M[i]), float(Mn[i])
        cam._keep = (R, cam_pos)
        cam.R, cam.cam_pos = R.data_ptr(), cam_pos.data_ptr()
        cam.width, cam.height = self.img_hw[1], self.img_hw[0]
        cam.row0, cam.row_step, cam.n_rows, cam.row_group = self.rows
        cam.radius = self.radius
        cam.n_views = self.n_views
        return cam

    def _coarse_steps(self):
        """(steps at 1/4 resolution, steps at 1/2 resolution) of the pyramid march (renderer.py:13,724-726)."""
        if list(self.scale_list) != [4, 2, 1] or len(self.march_step_list) != 3 or self.march_step_list[2] != -1:
            raise NotImplementedError("pyramid_recursive is implemented for scale_list=[4,2,1], march_step_list=[a,b,-1]")
        a, b = int(self.march_step_list[0]), int(self.march_step_list[1])
        if not (1 <= a <= 3 and 1 <= b <= 3 and a + b < self.march_step):
            raise NotImplementedError("pyramid_recursive: coarse step counts must be in [1,3]")
        return a, b

    def _coarse_dims(self):
        h, w = self.local_hw
        h1, w1 = (h + 1) // 2, (w + 1) // 2
        h2, w2 = (h1 + 1) // 2, (w1 + 1) // 2
        return (h1, w1), (h2, w2)

    def _coarse_homo(self):
        """K^-1 [xc, yc, 1] of the pooled pixel centres of the 1/2 and 1/4 resolution levels (renderer.py:604-636)."""
        if getattr(self, "_chomo", None) is None:
            res = []
            for (hh, ww), scale in zip(self._coarse_dims(), (2, 4)):
                # the `scale` fine rows pooled into one coarse row are consecutive image rows (bands: 4-row groups)
                ys = self._image_rows(scale * torch.arange(hh, device=self.device)).float() + (scale - 1) / 2
                xs = scale * torch.arange(ww, device=self.device).float() + (scale - 1) / 2
                Y, X = torch.meshgrid(ys, xs, indexing="ij")
                homo = torch.stack([X.reshape(-1), Y.reshape(-1), torch.ones(hh * ww, device=self.device)], 0)
                res.append((torch.matmul(self.K_inv, homo),))
            self._chomo = res
        return self._chomo

    def _scratch(self, pyramid=False):
        """Reusable (not saved-for-backward) per-renderer device scratch, stream-ordered."""
        if pyramid and self._scr is not None and self._scr.get("pyr_f") is None:
            (h1, w1), (h2, w2) = self._coarse_dims()
            npc = (h1 * w1 + h2 * w2) * self.n_views
            self._scr["pyr_f"] = torch.empty(23 * npc, device=self.device, dtype=torch.float32)
            self._scr["pyr_i"] = torch.empty(4 * npc + 8, device=self.device, dtype=torch.int32)
            self._scr["pyr_b"] = torch.empty(npc, device=self.device, dtype=torch.uint8)
        if self._scr is None:
            P, dev = self.P, self.device
            SEG = (P + 1 + 127) // 128 * 128      # capacity of one row segment of the query arrays (dist_b200.h)
            f32 = dict(device=dev, dtype=torch.float32)
            i32 = dict(device=dev, dtype=torch.int32)
            self._scr = {
                "ray": torch.empty(3, P, **f32), "entry": torch.empty(P, **f32), "exit_": torch.empty(P, **f32),
                "entry0": torch.empty(P, **f32), "pyr_f": None, "pyr_i": None, "pyr_b": None,
                "z": torch.empty(P, **f32), "list_a": torch.empty(2 * SEG, **i32), "list_b": torch.empty(2 * SEG, **i32),
                "pts": torch.empty(2, 2 * SEG, 3, **f32), "sdf": torch.empty(2 * SEG, **f32),
                "counts": torch.empty(2 * (self.march_step + 2), **i32),
                "view_stat": torch.zeros(self.n_views, 4, **i32),
                "n_idx": torch.empty(P, **i32), "n_pts": torch.empty(P, 3, **f32), "n_grad": torch.empty(P, 3, **f32),
                "n_cnt": torch.empty(1, **i32),
                # backward replay rows (at most P * buffer_size)
                "b_row": torch.empty(P * self.buffer_size, **i32), "b_pts": torch.empty(P * self.buffer_size, 3, **f32),
                "b_coef": torch.empty(P * self.buffer_size, **f32), "b_dpts": torch.empty(P * self.buffer_size, 3, **f32),
                "b_cnt": torch.empty(1, **i32),
                # two-tier precision: per-half-tile one-pass flags, the rays' previous sdf
                "seg_approx": torch.zeros(2 * SEG // 64, device=dev, dtype=torch.uint8), "sprev": torch.empty(P, **f32),
            }
            # mask cache: per-step slot bases, and the backward's list of rows replayed from the cache
            n_b = P * self.buffer_size
            self._scr.update(mask_base=torch.zeros(self.march_step + 3, **i32), bm_row=torch.empty(n_b, **i32),
                             bm_slot=torch.empty(n_b, **i32), bm_sdf=torch.empty(n_b, **f32), bm_coef=torch.empty(n_b, **f32),
                             bm_dpts=torch.empty(n_b, 3, **f32), bm_cnt=torch.empty(1, **i32))
            # the exact re-query rows of the forward pass live in the backward replay scratch (free until backward)
            self._scr.update(rq_idx=self._scr["b_row"], rq_pts=self._scr["b_pts"], rq_sdf=self._scr["b_coef"],
                             rq_cnt=self._scr["b_cnt"])
            if pyramid:
                return self._scratch(pyramid=True)
        return self._scr

    def _raise_if_empty(self, stat=None):
        """renderer.py:214-215.  Reads view_stat back from the device, i.e. waits for the enqueued march."""
        stat = self._last_counts.cpu() if stat is None else stat
        if int(stat[:, 3].max()) != 0:
            raise FloatingPointError("non-finite sdf during the march: the decoder's activations overflow the fp16 "
                                     "operands of the tensor-core engine for this latent; use engine='simt'")
        if int(stat[:, 0].min()) == 0:   # view_stat[v][0]: rays of view v alive at step 0
            raise ValueError('No valid depth.')

    def _n_codes(self, latent):
        """Latent codes of one call: n_views when a multi-view call gets one code per view (latent (V, L)), else 1."""
        if self.n_views > 1 and torch.is_tensor(latent) and latent.dim() == 2 and latent.shape[0] == self.n_views:
            return self.n_views
        return 1

    def reset_row_counter(self):
        self.rows_evaluated.zero_()
        self.rows_grad.zero_()
        self.tile_counters.zero_()

    def flops_per_row(self):
        """F = 2 * sum K_l N_l of the folded network (SURVEY.md 8d: 3,146,752 for the standard 8x512 spec)."""
        return 2 * sum(k * n for k, n in zip(self.plan.K, self.plan.N))

    # ---- rendering --------------------------------------------------------------------------------------------
    def render_depth(self, latent, R, T, clamp_dist=0.1, sample_index_type='min_abs', profile=False, no_grad=False,
                     no_grad_depth=False, no_grad_mask=False, no_grad_camera=False, ray_marching_type='recursive',
                     use_transform=True, check_empty=True):
        """(Zdepth[P], valid_mask[P] bool, min_sdf[P]) -- renderer.py:836-878.

        On a multi-view renderer (``_fused_child``: R (V,3,3), T (V,3)) ``no_grad_depth`` may be a sequence of V flags: the
        views are marched together, each with the depth-gradient semantics of its own flag (`render_warp` renders its
        second view with no_grad_depth=True, renderer_warp.py:109)."""
        if no_grad:
            no_grad_depth, no_grad_mask, no_grad_camera = True, True, True
        ngd_views = None
        if isinstance(no_grad_depth, (list, tuple)):
            if len(no_grad_depth) != self.n_views or self.n_views > 31:
                raise ValueError("no_grad_depth needs one flag per view (at most 31 views)")
            ngd_views = [bool(f) for f in no_grad_depth]
            no_grad_depth = all(ngd_views)
        if sample_index_type != 'min_abs':
            raise NotImplementedError("sample_index_type='%s' is not implemented (only 'min_abs')" % sample_index_type)
        if ray_marching_type == 'pyramid_recursive':
            self._coarse_steps()
            if not self.full_image and self.rows[3] % 4 != 0:
                raise NotImplementedError("pyramid_recursive on a row band needs bands of 4-row groups "
                                          "(rows=(row0,row_step,n_rows,4)); single-row bands use 'recursive'")
        if ray_marching_type not in _MARCH:
            raise ValueError('Error! Invalid type of ray marching: {}.'.format(ray_marching_type))  # renderer.py:834
        any_grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (latent, R, T))
        # which samples keep their camera graph (dist_march_t.cam_grad_levels): no_grad_camera only detaches the points
        # of ray_marching_recursive (renderer.py:536-537,543-544); ray_marching_trivial -- also the coarse levels of the
        # pyramid -- never does (renderer.py:481-484), a quirk the reference's gradients carry and these reproduce
        cam_levels = 3
        if no_grad_camera:
            cam_levels = {"recursive": 0, "pyramid_recursive": 2}.get(ray_marching_type, 3)
        opts = dict(kind=ray_marching_type, clamp_dist=clamp_dist, use_transform=use_transform, engine=self.engine,
                    want_depth_grad=any_grad and not no_grad_depth, want_mask_grad=any_grad and not no_grad_mask,
                    cam_levels=cam_levels if any_grad else 0,
                    # dist_march_t.replay_grad_rounding: bit 31 = every view, else one bit per view
                    replay=(sum(1 << v for v, f in enumerate(ngd_views) if not f) if ngd_views is not None
                            else (0 if no_grad_depth else -2147483648)))
        Zdepth, mask, min_sdf, hit = _RenderDepthFn.apply(latent, R, T, self, opts)
        if check_empty:
            self._raise_if_empty()
        if torch.is_grad_enabled() and (R.requires_grad or T.requires_grad):
            # renderer.py:842,863: the fill of rays missing the unit sphere stays differentiable w.r.t. the camera
            cam_pos = self.get_camera_location(R, T)
            d = self.get_distance_from_origin(cam_pos, self.get_camera_rays(R)).reshape(-1)
            min_sdf = torch.where(hit, min_sdf, d + self.threshold - self.radius)
        if no_grad_depth:
            Zdepth = Zdepth.detach()
        elif ngd_views is not None and any(ngd_views):
            Zv = Zdepth.reshape(self.n_views, self.Pv)
            Zdepth = torch.stack([Zv[v].detach() if f else Zv[v] for v, f in enumerate(ngd_views)], 0).reshape(-1)
        if no_grad_mask and not (R.requires_grad or T.requires_grad):
            min_sdf = min_sdf.detach()
        return Zdepth, mask.bool(), min_sdf

    def render_normal(self, latent, R, T, Zdepth, valid_mask, clamp_dist=0.1, MAX_POINTS=100000, no_grad=False,
                      normalize=True, use_transform=True):
        """Znormal (3, P): analytic decoder input-gradient at the hit points -- renderer.py:880-910.

        Autograd connectivity (SURVEY.md H6).  The input gradient of a ReLU / weight-norm decoder is
        (1 - sdf^2) * a with `a` piecewise constant in (xyz, latent), so:
          * normalize=True (default): the unit normal is piecewise constant -- the reference's graph through this
            tensor to latent / R / T carries exact zeros, and the tensor returned here carries no graph;
          * normalize=False with gradients enabled (and not no_grad): the factor (1 - sdf^2) does depend on latent and,
            through the hit point p = M^T (c + ray * z), on R and T (z detached, renderer.py:211-212).  It is attached
            as the value-neutral multiplier f(sdf) / f(sdf).detach() with f = d tanh-chain / d pre-activation, the sdf
            being re-queried differentiably on the hit rows (one extra forward row + one backward-replay row per hit
            pixel), which reproduces the reference's second-order term without a second-order graph."""
        with torch.cuda.device(self.device):
            Znormal, n_idx = self._render_normal_raw(latent, R, T, Zdepth, valid_mask, clamp_dist, normalize,
                                                     use_transform)
            want_graph = (not normalize) and (not no_grad) and torch.is_grad_enabled() and \
                any(t is not None and t.requires_grad for t in (latent, R, T))
            if not want_graph:
                return Znormal
            from .functional import decode_sdf
            idx = torch.nonzero(valid_mask.reshape(-1).bool()).reshape(-1)
            if idx.numel() == 0:
                return Znormal
            v = idx // self.Pv if R.dim() == 3 else None
            cam_pos, cam_rays = self.get_camera_location(R, T), self.get_camera_rays(R)
            if v is None:
                pts = cam_rays[:, idx] * Zdepth.detach()[idx][None, :] + cam_pos[:, None]
            else:   # stacked poses: (V,3,Pv) rays, (V,3) centres
                pts = cam_rays[v, :, idx - v * self.Pv].t() * Zdepth.detach()[idx][None, :] + cam_pos[v].t()
            if use_transform:
                pts = self.inv_transform_points(pts)
            # one code per view: each hit row is decoded with its view's code
            index = v if (v is not None and self._n_codes(latent) > 1) else None
            o = decode_sdf(self.decoder, latent, pts.t(), clamp_dist=None, engine=self.engine,
                           latent_index=index).squeeze(-1)

            def dchain(x):     # d sdf / d pre-activation as a function of the sdf value (deep_sdf_decoder.py:99-110)
                if self.plan.use_tanh:
                    return (1 - x * x) * (1 - torch.atanh(x) ** 2)
                return 1 - x * x
            factor = dchain(o) / dchain(o.detach())
            scale = torch.ones(self.P, device=self.device, dtype=torch.float32).index_copy(0, idx, factor)
            return Znormal * scale[None, :]

    def _render_normal_raw(self, latent, R, T, Zdepth, valid_mask, clamp_dist, normalize, use_transform):
        lib, st = _abi.lib(), _stream(self.device)
        plan = self.plan
        plan.refresh()
        engine = resolve_engine(plan, self.engine)
        net, engine, _keep = plan.net_for(latent, engine, st, n_codes=self._n_codes(latent))
        Rd = R.detach().float().contiguous()
        cam_pos = self.get_camera_location(Rd, T.detach().float()).contiguous()
        cam = self._c_camera(Rd, cam_pos, use_transform)
        scr = self._scratch()
        Zd = Zdepth.detach().float().contiguous()
        m8 = valid_mask.detach().to(torch.uint8).contiguous()
        Znormal = torch.empty(3, self.P, device=self.device, dtype=torch.float32)
        _abi.check(lib.dist_render_normal_fwd(net, engine, cam, _abi.ptr(Zd), _abi.ptr(m8), float(clamp_dist),
                                              1 if normalize else 0, _abi.ptr(Znormal), _abi.ptr(scr["n_idx"]),
                                              _abi.ptr(scr["n_pts"]), _abi.ptr(scr["n_grad"]), _abi.ptr(scr["n_cnt"]),
                                              _abi.ptr(self.rows_grad), st))
        return Znormal, scr["n_idx"]

    def render(self, latent, R, T, clamp_dist=0.1, sample_index_type='min_abs', profile=False, no_grad=False,
               no_grad_depth=False, no_grad_normal=False, no_grad_mask=False, no_grad_camera=False,
               normalize_normal=True, use_transform=True, ray_marching_type='pyramid_recursive',
               num_forward_sampling=0, check_empty=True):
        """(depth[h,w], normal[h,w,3], mask[h,w] uint8, min_abs_query[h,w]) -- renderer.py:943-999."""
        if no_grad:
            no_grad_depth, no_grad_normal, no_grad_mask, no_grad_camera = True, True, True, True
        h, w = self.local_hw
        Zdepth, valid_mask, min_abs_query = self.render_depth(
            latent, R, T, clamp_dist=clamp_dist, sample_index_type=sample_index_type, profile=profile, no_grad=no_grad,
            no_grad_depth=no_grad_depth, no_grad_mask=no_grad_mask, no_grad_camera=no_grad_camera,
            ray_marching_type=ray_marching_type, use_transform=use_transform, check_empty=False)
        V, stacked = self.n_views, R.dim() == 3
        calib = self.calib_map.repeat(V) if stacked else self.calib_map
        depth = torch.where(valid_mask, Zdepth * calib, torch.full_like(Zdepth, 1e11))  # renderer.py:967-969
        if self.use_depth2normal:
            # renderer.py:972-975: normals by central differences of the depth map; like the reference's helper this
            # zeroes the background of the returned depth map in place (render_utils.py:24-25)
            from .render_utils import depth2normal
            fx, fy = np.float32(self.intrinsic[0, 0]), np.float32(self.intrinsic[1, 1])
            dmap = depth.reshape((V, h, w) if stacked else (h, w))
            normal = torch.stack([depth2normal(dmap[v], fx, fy) for v in range(V)], 0) if stacked \
                else depth2normal(dmap, fx, fy)
            out = (dmap, normal, valid_mask.reshape(dmap.shape).type(torch.uint8), min_abs_query.reshape(dmap.shape))
            if num_forward_sampling != 0:
                if stacked:
                    raise NotImplementedError("forward sampling is not available on the multi-view march")
                inside = self.forward_sampling(latent, R, T, Zdepth, valid_mask, clamp_dist=clamp_dist,
                                               num_forward_sampling=num_forward_sampling, use_transform=use_transform)
                out = out + (inside.reshape(h, w, num_forward_sampling),)
            if check_empty:
                self._raise_if_empty()
            return out
        normal = self.render_normal(latent, R, T, Zdepth, valid_mask, clamp_dist=clamp_dist, no_grad=no_grad_normal,
                                    normalize=normalize_normal, use_transform=use_transform)
        if stacked:     # a stack of poses marched together (render_views): maps get a leading view axis
            if num_forward_sampling != 0:
                raise NotImplementedError("forward sampling is not available on the multi-view march")
            # pose by pose with the single-pose GEMM on contiguous operands: a batched GEMM may round differently
            Rn, n3 = R, normal.reshape(3, V, -1)   # renderer.py:977-978: no_grad_normal detaches Znormal, never R
            normal = torch.stack([torch.matmul(Rn[v], n3[:, v].contiguous()) for v in range(V)], 0)   # renderer.py:978
            normal = torch.cat([normal[:, :1] * (-1), normal[:, 1:]], 1).reshape(V, 3, h, w).permute(0, 2, 3, 1)
            out = (depth.reshape(V, h, w), normal, valid_mask.reshape(V, h, w).type(torch.uint8),
                   min_abs_query.reshape(V, h, w))
            if check_empty:
                self._raise_if_empty()
            return out
        normal = torch.matmul(R, normal)  # renderer.py:978 (no_grad_normal detaches Znormal only, renderer.py:909)
        normal = torch.cat([normal[:1] * (-1), normal[1:]], 0)                   # renderer.py:979
        normal = normal.reshape(3, h, w).permute(1, 2, 0)
        out = (depth.reshape(h, w), normal, valid_mask.reshape(h, w).type(torch.uint8), min_abs_query.reshape(h, w))
        if num_forward_sampling != 0:   # renderer.py:984-986
            inside = self.forward_sampling(latent, R, T, Zdepth, valid_mask, clamp_dist=clamp_dist,
                                           num_forward_sampling=num_forward_sampling, use_transform=use_transform)
            out = out + (inside.reshape(h, w, num_forward_sampling),)
        if check_empty:
            self._raise_if_empty()   # deferred to here so that the whole render is enqueued before the host waits
        return out

    # ---- multi-view batching ------------------------------------------------------------------------------------
    def _fused_child(self, V):
        """Shallow copy of this renderer that marches V views of the same shape in ONE call (n_views = V): private
        scratch sized for V * Pv pixels, everything else shared."""
        import copy
        cache = self.__dict__.setdefault("_fused", {})
        child = cache.get(V)
        if child is None:
            child = copy.copy(self)
            child.n_views, child.P = V, V * self.Pv
            child._scr, child._last_counts, child._slots, child._fused = None, None, None, {}
            cache[V] = child
        return child

    def _view_slots(self, n):
        """n (stream, renderer) pairs: shallow copies of this renderer with private scratch, one CUDA stream each."""
        import copy
        slots = getattr(self, "_slots", None) or []
        while len(slots) < n:
            child = copy.copy(self)
            child._scr, child._last_counts, child._slots, child._fused = None, None, None, {}
            slots.append((torch.cuda.Stream(device=self.device), child))
        self._slots = slots
        return slots[:n]

    def render_views(self, latent, Rs, Ts, fused=True, n_streams=1, **kw):
        """``render()`` of V camera poses, batched: returns the outputs of ``render`` stacked along a new leading view
        axis -- (depth[V,h,w], normal[V,h,w,3], mask[V,h,w] uint8, min_abs_query[V,h,w]).

        ``latent``: one code shared by every view, (1, L) or (L,), or one code per view, (V, L) -- view v is then
        rendered with ``latent[v]``, exactly as ``render(latent[v], Rs[v], Ts[v])`` renders it, and the gradient reaches
        ``latent`` as (V, L).  So S shapes (or shapes x poses, ``render_views(codes[shape_of_view], Rs, Ts)``) march
        together and pay the per-step cost of the march tail once.  (An extension: the reference renders one code per
        call.)

        The multi-view callers of the reference (`optimize_multi.py:62-80`, `renderer_warp.py:108-109`) render their
        views one after the other and synchronise with the host several times per march step.

        ``fused=True`` (default): ONE march over all V * h * w rays (`dist_camera_t.n_views`): one compaction list, one
        decoder launch per step, one normal launch, one backward replay.  The long tail of a march -- dozens of
        launches that keep a few SM pairs busy for one tile latency each while the last grazing rays converge -- is
        paid once instead of V times.  Every view keeps the per-render semantics of the reference (own early break,
        own 'No valid depth' test, own pyramid levels), so the maps are those of V separate ``render`` calls bit for
        bit; gradients reach ``latent``, ``Rs``, ``Ts`` as usual.
        ``fused=False`` (or ``num_forward_sampling != 0``): the views are enqueued one after the other without host
        synchronisation, optionally round-robin on ``n_streams`` CUDA streams with private scratch."""
        check_empty = kw.pop("check_empty", True)
        V = len(Rs)
        if V == 0 or len(Ts) != V:
            raise ValueError("render_views needs V >= 1 rotations and as many translations")
        per_view = False
        if torch.is_tensor(latent) and latent.dim() == 2 and latent.shape[0] != 1:
            if latent.shape[0] != V:
                raise ValueError("latent must be (1, L), (L,) or one code per view (%d, L); got %s"
                                 % (V, tuple(latent.shape)))
            per_view = True
        if fused and kw.get("num_forward_sampling", 0) == 0:
            R = Rs if torch.is_tensor(Rs) else torch.stack(list(Rs), 0)
            T = Ts if torch.is_tensor(Ts) else torch.stack(list(Ts), 0)
            return self._fused_child(V).render(latent, R, T, check_empty=check_empty, **kw)
        main = torch.cuda.current_stream(self.device)
        # lazily built caches are created on this stream before any view stream can touch them
        _ = self.calib_map, self._coarse_homo()
        self.plan.refresh()
        self.plan.net_for(latent[:1] if per_view else latent, resolve_engine(self.plan, self.engine),
                          main.cuda_stream)  # one-time engine preparation
        n_streams = max(1, min(int(n_streams), V))
        slots = self._view_slots(n_streams)
        side = n_streams > 1
        n_valid = torch.empty(V, device=self.device, dtype=torch.int32)
        if side:
            for st, _ in slots:
                st.wait_stream(main)
        outs = []
        for v in range(V):
            st, child = slots[v % n_streams]
            with torch.cuda.stream(st if side else main):
                o = child.render(latent[v] if per_view else latent, Rs[v], Ts[v], check_empty=False, **kw)
                n_valid[v:v + 1].copy_(child._last_counts[:, 0])
            outs.append(o)
        if side:
            for st, _ in slots:
                main.wait_stream(st)
            for o in outs:
                for t in o:
                    t.record_stream(main)
        res = tuple(torch.stack([o[i] for o in outs], 0) for i in range(len(outs[0])))
        if check_empty and min(n_valid.tolist()) == 0:
            raise ValueError('No valid depth.')
        return res

    def forward_sampling(self, latent, R, T, Zdepth, valid_mask, clamp_dist=0.1, num_forward_sampling=1, no_grad=False,
                         use_transform=True):
        """sdf + offset at points pushed `offset` beyond the hit point along the ray (renderer.py:912-941), (P, k).
        The decoder rows go through decode_sdf (CUDA engines); differentiable w.r.t. latent and the camera."""
        from .functional import decode_sdf
        assert num_forward_sampling > 0
        cam_pos = self.get_camera_location(R, T)
        cam_rays = self.get_camera_rays(R)
        inside = torch.zeros(self.P, num_forward_sampling, device=self.device, dtype=torch.float32)
        valid_mask = valid_mask.bool()
        idx = torch.nonzero(valid_mask).reshape(-1)
        if idx.numel() == 0:
            return inside
        rays_v, z_v = cam_rays[:, idx], Zdepth[idx]
        cols = []
        for i in range(num_forward_sampling):
            grid = 0.5 * clamp_dist * (i + 1) / num_forward_sampling
            pts = self.generate_point_samples(cam_pos, rays_v, z_v + grid, has_zdepth_grad=False, inv_transform=use_transform)
            sdf = decode_sdf(self.decoder, latent, pts.transpose(1, 0), clamp_dist=None, no_grad=no_grad,
                             engine=self.engine).squeeze(-1)
            cols.append(sdf[:, None] + grid)
        return inside.index_copy(0, idx, torch.cat(cols, 1))

    def render_silhouette(self, latent, R, T, **kw):
        """(mask[h,w] uint8, min_abs_query[h,w]): the pair the reference uses as the silhouette (renderer.py:878,990)."""
        h, w = self.local_hw
        _, valid_mask, min_abs_query = self.render_depth(latent, R, T, **kw)
        return valid_mask.reshape(h, w).type(torch.uint8), min_abs_query.reshape(h, w)
