"""GPU: several shapes in one fused march -- one latent code per view in render_views, one code per row in decode_sdf
(latent_index).  Each view / row must be what a call with its own code alone computes: maps and decoder outputs bit for
bit, gradients to the rounding of their atomic sums."""
import importlib

import pytest
import torch

import cases
import gpu_util as gu

pytestmark = pytest.mark.gpu
pkg = cases.pkg
synth = cases.synth
plan_for = importlib.import_module("dist-renderer_b200.plan").plan_for
resolve_engine = importlib.import_module("dist-renderer_b200.functional").resolve_engine

HW = (48, 40)
V = 5
KINDS = ("recursive", "pyramid_recursive", "trivial")


def _codes(n, seed0=20):
    return torch.cat([synth.make_latent(seed=seed0 + i) for i in range(n)], 0).cuda()


@pytest.fixture(scope="module")
def dec():
    return gu.gpu_decoder("B")


@pytest.fixture(scope="module")
def views():
    ring = synth.ring_cameras(24, 25.0, 2.5)[::5][:V]
    return torch.stack([R for R, _ in ring]).cuda(), torch.stack([T for _, T in ring]).cuda()


def _renderer(dec, **kw):
    return pkg.SDFRenderer(dec, synth.intrinsic(*HW, focal_scale=1.2 * 2.5 / 1.6), img_hw=HW, march_step=50,
                           buffer_size=5, **kw)


def _separate(ren, codes, Rs, Ts, **kw):
    """V independent render() calls, view v with codes[v]: maps and the gradients of the summed loss."""
    lat = codes.clone().requires_grad_(True)
    Rg, Tg = Rs.clone().requires_grad_(True), Ts.clone().requires_grad_(True)
    outs = [ren.render(lat[v], Rg[v], Tg[v], **kw) for v in range(len(codes))]
    sum(cases.scalar_loss(o) for o in outs).backward()
    return outs, (lat.grad, Rg.grad, Tg.grad)


def _batched(ren, codes, Rs, Ts, **kw):
    lat = codes.clone().requires_grad_(True)
    Rg, Tg = Rs.clone().requires_grad_(True), Ts.clone().requires_grad_(True)
    out = ren.render_views(lat, Rg, Tg, **kw)
    sum(cases.scalar_loss(tuple(b[v] for b in out)) for v in range(len(codes))).backward()
    return out, (lat.grad, Rg.grad, Tg.grad)


def _assert_same(outs, batched, grads_a, grads_b, what):
    bad = [(what, v, name, float((a.detach().float() - b[v].detach().float()).abs().max()))
           for v, o in enumerate(outs) for name, a, b in zip(("depth", "normal", "mask", "min_sdf"), o, batched)
           if not torch.equal(a.detach(), b[v].detach())]
    assert not bad, bad
    assert grads_b[0].shape == grads_a[0].shape
    for name, x, y in zip(("latent", "R", "T"), grads_b, grads_a):
        assert gu.rel(x, y) < 1e-5, (what, name, gu.rel(x, y))


def test_fold_of_several_codes_equals_single_folds(dec):
    """dist_fold_latent with n_codes = C: row c of both tables (and the tensor-core engine's scaled copy) is byte for
    byte the single-code fold of code c."""
    plan = plan_for(dec)
    C = 5
    codes = _codes(C)
    st = torch.cuda.current_stream().cuda_stream
    for engine in ("tc", "simt"):
        eng = resolve_engine(plan, engine)
        _, eng, (b0, bl, bl_tc, _) = plan.net_for(codes, eng, st, n_codes=C)
        for c in range(C):
            _, _, (s0, sl, sl_tc, _) = plan.net_for(codes[c:c + 1], eng, st)
            n0, nl = s0.numel(), sl.numel()
            assert b0.numel() == C * n0 and bl.numel() == C * nl
            assert torch.equal(b0[c * n0:(c + 1) * n0], s0) and torch.equal(bl[c * nl:(c + 1) * nl], sl)
            if engine == "tc":
                assert torch.equal(bl_tc[c * nl:(c + 1) * nl], sl_tc)


@pytest.mark.parametrize("engine", ["tc", "simt"])
def test_decode_sdf_latent_index(dec, engine):
    """Rows with codes assigned at random (mixed warps and tiles, one code without rows) equal per-code calls; the
    gradient reaches (C, L) and the points, and the code without rows gets an exact zero."""
    C, n = 5, 10000
    g = torch.Generator().manual_seed(7)
    codes = _codes(C)
    pts = ((torch.rand(n, 3, generator=g) - 0.5) * 1.4).cuda()
    idx = torch.randint(0, C, (n,), generator=g)
    idx[idx == 3] = 1                                   # code 3: no rows
    idx = idx.cuda()
    w = torch.randn(n, generator=g).cuda()
    for index, label in ((idx, "mixed"), (torch.full((n,), 2, dtype=torch.long, device="cuda"), "one code")):
        out = pkg.decode_sdf(dec, codes, pts, latent_index=index, engine=engine, no_grad=True)
        assert out.shape == (n, 1)
        for c in range(C):
            sel = index == c
            if bool(sel.any()):
                ref = pkg.decode_sdf(dec, codes[c:c + 1], pts[sel], engine=engine, no_grad=True)
                assert torch.equal(out[sel], ref), (label, c)
        lat, p = codes.clone().requires_grad_(True), pts.clone().requires_grad_(True)
        (pkg.decode_sdf(dec, lat, p, clamp_dist=None, latent_index=index, engine=engine).squeeze(-1) * w).sum().backward()
        assert lat.grad.shape == (C, codes.shape[1])
        for c in range(C):
            sel = index == c
            if not bool(sel.any()):
                assert bool((lat.grad[c] == 0).all()), (label, c)
                continue
            lc, pc = codes[c:c + 1].clone().requires_grad_(True), pts[sel].clone().requires_grad_(True)
            (pkg.decode_sdf(dec, lc, pc, clamp_dist=None, engine=engine).squeeze(-1) * w[sel]).sum().backward()
            assert gu.rel(lat.grad[c], lc.grad[0]) < 1e-5, (label, c, gu.rel(lat.grad[c], lc.grad[0]))
            assert gu.rel(p.grad[sel], pc.grad) < 1e-5, (label, c)


@pytest.mark.parametrize("kind", KINDS)
def test_render_views_per_view_codes(dec, views, kind):
    """V views, each with its own code, fused and looped: maps bit-identical to V separate renders, gradients
    (latent (V, L), Rs, Ts) to rel 1e-5."""
    Rs, Ts = views
    codes = _codes(V)
    ren = _renderer(dec)
    outs, g_sep = _separate(ren, codes, Rs, Ts, ray_marching_type=kind)
    for mode in (dict(fused=True), dict(fused=False, n_streams=2)):
        out, g = _batched(ren, codes, Rs, Ts, ray_marching_type=kind, **mode)
        assert out[0].shape == (V,) + HW and out[1].shape == (V,) + HW + (3,) and out[2].dtype == torch.uint8
        _assert_same(outs, out, g_sep, g, (kind, mode))


@pytest.mark.parametrize("variant", [dict(engine="simt"), dict(screen=False, mask_cache=False)])
def test_render_views_per_view_codes_variants(dec, views, variant):
    """The same on the fp32 engine, and on the tensor-core engine with one precision tier and no mask cache."""
    Rs, Ts = views
    codes = _codes(V)
    ren = _renderer(dec, **variant)
    for kind in ("recursive", "pyramid_recursive"):
        outs, g_sep = _separate(ren, codes, Rs, Ts, ray_marching_type=kind)
        out, g = _batched(ren, codes, Rs, Ts, ray_marching_type=kind)
        _assert_same(outs, out, g_sep, g, (kind, variant))


def test_shared_code_written_out_per_view(dec, views):
    """latent.expand(V, L) takes the per-view path and gives the shared-code maps; autograd sums its gradient."""
    Rs, Ts = views
    ren = _renderer(dec)
    for kind in ("recursive", "pyramid_recursive"):
        la = synth.make_latent().cuda().requires_grad_(True)
        a = ren.render_views(la, Rs, Ts, ray_marching_type=kind)
        sum(cases.scalar_loss(tuple(x[v] for x in a)) for v in range(V)).backward()
        lb = synth.make_latent().cuda().requires_grad_(True)
        b = ren.render_views(lb.expand(V, lb.shape[1]), Rs, Ts, ray_marching_type=kind)
        sum(cases.scalar_loss(tuple(x[v] for x in b)) for v in range(V)).backward()
        assert all(torch.equal(x.detach(), y.detach()) for x, y in zip(a, b)), kind
        assert lb.grad.shape == la.grad.shape and gu.rel(lb.grad, la.grad) < 1e-5, (kind, gu.rel(lb.grad, la.grad))


def test_unnormalized_normals_per_view_codes(dec, views):
    """normalize_normal=False keeps its graph term with per-view codes (decode_sdf with latent_index on the hit rows)."""
    Rs, Ts = views
    codes = _codes(V)
    ren = _renderer(dec)
    outs, g_sep = _separate(ren, codes, Rs, Ts, ray_marching_type="recursive", normalize_normal=False)
    out, g = _batched(ren, codes, Rs, Ts, ray_marching_type="recursive", normalize_normal=False)
    _assert_same(outs, out, g_sep, g, "normalize_normal=False")


def _loss_mix(out, gt):
    """Depth / normal / silhouette mix in the spirit of loss_single.compute_all_loss (weights 10/5/1)."""
    depth, normal, mask, min_sdf = out
    gdepth, gnormal, gmask = gt
    both = mask.bool() & gmask.bool()
    l_depth = (depth[both] - gdepth[both]).abs().mean() if bool(both.any()) else depth.sum() * 0
    l_normal = (1 - (normal[both] * gnormal[both]).sum(-1)).mean() if bool(both.any()) else normal.sum() * 0
    inside = gmask.bool()
    l_mask = torch.relu(min_sdf[inside]).mean() + torch.relu(-min_sdf[~inside] + 1e-3).mean()
    return 10.0 * l_depth + 5.0 * l_normal + 1.0 * l_mask


def test_batched_shape_optimisation_tracks_independent_loops(dec):
    """S shape codes optimised together (Adam on (S, L), one render_views per iteration) follow the loss trajectories of
    S independent single-shape loops."""
    S, hw, n_it = 4, (32, 32), 6
    K, (R, T) = synth.intrinsic(*hw), synth.lookat_camera(30.0, 20.0, 1.6)
    R, T = R.cuda(), T.cuda()
    ren = pkg.SDFRenderer(dec, K, img_hw=hw, march_step=60, buffer_size=3)
    gts = [[t.detach() for t in ren.render(synth.make_latent(seed=40 + s).cuda(), R, T, no_grad=True)[:3]]
           for s in range(S)]
    init = _codes(S, seed0=50)

    def independent(s):
        lat = init[s:s + 1].clone().requires_grad_(True)
        opt = torch.optim.Adam([lat], lr=1e-3)
        losses = []
        for _ in range(n_it):
            opt.zero_grad()
            loss = _loss_mix(ren.render(lat, R, T), gts[s])
            loss.backward()
            opt.step()
            losses.append(float(loss.detach()))
        return losses
    ref = [independent(s) for s in range(S)]
    lat = init.clone().requires_grad_(True)
    opt = torch.optim.Adam([lat], lr=1e-3)
    Rs, Ts = R.expand(S, 3, 3).contiguous(), T.expand(S, 3).contiguous()
    got = [[] for _ in range(S)]
    for _ in range(n_it):
        opt.zero_grad()
        out = ren.render_views(lat, Rs, Ts)
        per_shape = [_loss_mix(tuple(x[s] for x in out), gts[s]) for s in range(S)]
        sum(per_shape).backward()
        opt.step()
        for s in range(S):
            got[s].append(float(per_shape[s]))
    print("independent", ref, "batched", got)
    for s in range(S):
        for a, b in zip(got[s], ref[s]):
            assert abs(a - b) <= 2e-3 * abs(b) + 1e-6, (s, got[s], ref[s])


def test_errors(dec, views):
    Rs, Ts = views
    ren = _renderer(dec)
    with pytest.raises(ValueError):
        ren.render_views(_codes(V + 1), Rs, Ts, no_grad=True)
    with pytest.raises(ValueError):
        ren.render_views(_codes(V + 1), Rs, Ts, fused=False, no_grad=True)
    # one view whose rays all pass far from the unit sphere: 'No valid depth', whichever way the views are executed
    R_away, T_away = Rs.clone(), Ts.clone()
    R_away[2], T_away[2] = torch.eye(3).cuda(), torch.tensor([50.0, 0.0, 1.6]).cuda()
    for mode in (dict(fused=True), dict(fused=False)):
        with pytest.raises(ValueError, match="No valid depth"):
            ren.render_views(_codes(V), R_away, T_away, ray_marching_type="recursive", no_grad=True, **mode)
    codes = _codes(3)
    pts = (torch.rand(100, 3) - 0.5).cuda()
    for bad in (torch.full((100,), 3, dtype=torch.long), torch.full((100,), -1, dtype=torch.long),
                torch.zeros(99, dtype=torch.long), torch.zeros(100, dtype=torch.float32)):
        with pytest.raises(ValueError):
            pkg.decode_sdf(dec, codes, pts, latent_index=bad.cuda())
