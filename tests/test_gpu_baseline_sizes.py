"""GPU: parity at the sizes BASELINE.json names and on every gradient flag, against fixtures written by the REAL
reference (oracle/make_golden.py --big / --flags), on the tensor-core engine (the product default).

Gate (BASELINE.md section 3): depth rel-L2 <= 1e-4 on the mask intersection; mask XOR reported and bounded by the
fp32-vs-fp64 floor of the reference itself; min_sdf rel-L2 <= 1e-4 (split into converged / unconverged pixels, the
plain figure over all P printed beside it); normal rel-L2 <= 1e-4 after excluding ReLU-flip outlier pixels;
d latent / dR / dT rel-L2.  The deviation of the reference's fp64 twin from the fp32 reference (stored in the
fixture) is printed beside every number as the noise floor.
"""
import importlib
import os

import numpy as np
import pytest
import torch

import cases
import gpu_util as gu

pytestmark = pytest.mark.gpu
pkg = cases.pkg
synth = cases.synth
par = importlib.import_module("dist-renderer_b200.parallel")


def _gold(name):
    return np.load(os.path.join(cases.GOLDEN_DIR, name + ".npz"))


def _ref_of(gold):
    ref = [torch.from_numpy(gold[k]) for k in ("depth", "normal", "mask", "min_sdf")]
    gref = [torch.from_numpy(gold[k]) for k in ("g_latent", "g_R", "g_T")]
    return ref, gref


@pytest.mark.parametrize("name", sorted(cases.BIG_CASES))
def test_baseline_size_matches_reference_golden(name):
    """A fixture with `pix` holds depth / normal / min_sdf at that seeded sample of pixels only (the mask whole, and its
    floor measured on the same pixels): the maps are compared there, the mask XOR over the whole image."""
    cs = cases.BIG_CASES[name]
    gold = _gold("big_" + name)
    floor = dict(zip(gold["floor_keys"].tolist(), gold["floor_vals"].tolist()))
    out, g, ren = gu.run_gpu(cs, engine="tc")
    ref, gref = _ref_of(gold)
    xor = int((out[2] != ref[2]).sum())
    if "pix" in gold.files:
        out, ref[2] = gu.at_pixels(out, gold["pix"]), gu.at_pixels([ref[2]], gold["pix"])[0]
    res = gu.measure(out, ref, g, gref)
    res["xor"] = xor
    print("\n%s  (P = %d, hits %d)" % (name, ref[2].numel(), res["hits"]))
    for k in ("xor", "depth", "normal", "n_out", "min_sdf", "min_sdf_converged_maxabs", "min_sdf_all_P", "g_latent",
              "g_R", "g_T"):
        print("  %-26s tc-vs-reference %-12.4g reference-fp64-twin floor %.4g" % (k, res[k], floor.get(k, float("nan"))))
    # mask: threshold-adjacent rays flip under ANY change of rounding; the reference's own fp64 twin flips floor["xor"]
    assert res["xor"] <= max(4, 2 * int(floor["xor"]) + 4), res
    assert res["depth"] < 1e-4 and res["min_sdf"] < 1e-4 and res["min_sdf_converged_maxabs"] <= 1e-4, res
    # normals: <= 1e-4 after excluding ReLU-flip outlier pixels.  How many pixels flip is a property of the hit points'
    # last bits: the reference's own fp64 twin flips floor["n_out"] of them; a faithful fp32 render lands within a small
    # multiple of that (SURVEY H2 proposes 2x; counts of 5-30 pixels fluctuate, so 3x here) or the 0.1 % bar, printed above
    assert res["normal"] < 1e-4, res
    assert res["n_out"] <= max(3 * int(floor["n_out"]), res["n_out_strict_allowed"]), (res, floor)
    # a flipped silhouette pixel moves sum(depth) by a whole depth value: gradients are compared at the fp64 floor's scale
    gtol = 2e-3 if res["xor"] == 0 else 3e-2
    for k in ("g_latent", "g_R", "g_T"):
        assert res[k] < max(gtol, 3 * floor[k]), (k, res, floor)


@pytest.mark.parametrize("engine", ["simt", "tc"])
@pytest.mark.parametrize("name", sorted(cases.FLAG_CASES))
def test_gradient_flags_match_reference_golden(name, engine):
    """render() under each no_grad_* / normalize_normal flag (renderer.py:943-957): outputs and the gradients that
    survive the flag, including the reference's quirk that the coarse pyramid levels ignore no_grad_camera."""
    cs = cases.FLAG_CASES[name]
    gold = _gold(name)
    dev = torch.device("cuda")
    dec = gu.gpu_decoder(cs["decoder"])
    K, R, T = cases.camera(cs["cam"], cs["hw"])
    ren = pkg.SDFRenderer(dec, K, img_hw=cs["hw"], march_step=cs["march_step"], buffer_size=cs["buffer_size"], engine=engine)
    lat = synth.make_latent().to(dev).requires_grad_(True)
    Rg, Tg = R.to(dev).requires_grad_(True), T.to(dev).requires_grad_(True)
    out = ren.render(lat, Rg, Tg, ray_marching_type=cs["kind"], **cs["flags"])
    cases.scalar_loss(out).backward()
    g = [t.grad.cpu() if t.grad is not None else torch.zeros(t.shape) for t in (lat, Rg, Tg)]
    ref, gref = _ref_of(gold)
    out = [o.detach().cpu() for o in out]
    res = gu.measure(out, ref)
    assert res["xor"] <= 2 and res["depth"] < 1e-4 and res["min_sdf"] < 1e-4, res
    if cs["flags"].get("normalize_normal", True):
        assert res["normal"] < 1e-4 and res["n_out"] <= res["n_allowed"], res
    else:   # un-normalised normals: gradient magnitudes, compared pixel-wise relative to their own norm
        m = out[2].bool() & ref[2].bool()
        e = (out[1][m] - ref[1][m]).norm(dim=-1) / ref[1][m].norm(dim=-1)
        assert int((e > 1e-3).sum()) <= max(3, int(0.005 * int(m.sum()))), float(e.max())
    for name_g, a, b in zip(("g_latent", "g_R", "g_T"), g, gref):
        if float(b.abs().max()) < 1e-6:
            assert float(a.abs().max()) < 1e-6, (name_g, float(a.abs().max()))     # the flag cuts this gradient
        else:
            assert gu.rel(a, b) < (2e-3 if res["xor"] == 0 else 3e-2), (name_g, gu.rel(a, b), res)


@pytest.mark.parametrize("engine", ["simt", "tc"])
def test_render_silhouette_matches_reference_golden(engine):
    """render_silhouette = the (valid_mask, min_sdf) pair of the reference's render_depth (renderer.py:878)."""
    cs = cases._FLAG_BASE
    gold = _gold("silhouette_48")
    dev = torch.device("cuda")
    K, R, T = cases.camera(cs["cam"], cs["hw"])
    ren = pkg.SDFRenderer(gu.gpu_decoder("B"), K, img_hw=cs["hw"], march_step=cs["march_step"],
                          buffer_size=cs["buffer_size"], engine=engine)
    lat = synth.make_latent().to(dev).requires_grad_(True)
    Rg, Tg = R.to(dev).requires_grad_(True), T.to(dev).requires_grad_(True)
    mask, min_sdf = ren.render_silhouette(lat, Rg, Tg, ray_marching_type=cs["kind"])
    assert mask.shape == cs["hw"] and mask.dtype == torch.uint8 and min_sdf.shape == cs["hw"]
    min_sdf.sum().backward()
    assert int((mask.cpu() != torch.from_numpy(gold["mask"]).to(torch.uint8)).sum()) <= 2
    a, b = min_sdf.detach().cpu().reshape(-1).double(), torch.from_numpy(gold["min_sdf"]).reshape(-1).double()
    conv = (a.abs() <= 5e-5) & (b.abs() <= 5e-5)
    assert gu.rel(a[~conv], b[~conv]) < 1e-4 and float((a[conv] - b[conv]).abs().max()) <= 1e-4
    for t, key in zip((lat, Rg, Tg), ("g_latent", "g_R", "g_T")):
        assert gu.rel(t.grad.cpu(), gold[key]) < 2e-3, key


@pytest.mark.parametrize("engine", ["simt", "tc"])
@pytest.mark.parametrize("name", ["earlybreak_recursive_16", "earlybreak_pyramid_16"])
def test_earlybreak_padding_render_depth(name, engine):
    """renderer.py:562-567 (padding with copies of the last step when the march breaks before buffer_size steps), also
    for the full-resolution level of the pyramid march: raw Zdepth of render_depth and the gradient through all
    buffer_size selected samples, against the reference."""
    cs = cases.CASES[name]
    gold = _gold(name)
    dev = torch.device("cuda")
    K, R, T = cases.camera(cs["cam"], cs["hw"])
    ren = pkg.SDFRenderer(gu.gpu_decoder("B"), K, img_hw=cs["hw"], march_step=cs["march_step"],
                          buffer_size=cs["buffer_size"], engine=engine)
    lat = synth.make_latent().to(dev).requires_grad_(True)
    Rg, Tg = R.to(dev).requires_grad_(True), T.to(dev).requires_grad_(True)
    Zd, _, _ = ren.render_depth(lat, Rg, Tg, ray_marching_type=cs["kind"])
    Zd[Zd < 1e10].sum().backward()
    ref = torch.from_numpy(gold["rd_Zdepth"])
    hit = ref < 1e10
    assert bool(((Zd.detach().cpu() < 1e10) == hit).all())
    assert gu.rel(Zd.detach().cpu()[hit], ref[hit]) < 1e-5
    for t, key in zip((lat, Rg, Tg), ("rd_g_latent", "rd_g_R", "rd_g_T")):
        assert gu.rel(t.grad.cpu(), gold[key]) < 2e-3, key


@pytest.mark.parametrize("kind", ["recursive", "pyramid_recursive"])
def test_config5_2048_bands_equal_full_image(kind):
    """Config 5 (2048 x 2048, forward depth + normal): the image rendered as 8 interleaved bands of 4-row groups -- what 8
    ranks render -- equals the full-image render bit for bit, for the reference's default pyramid march too; and the
    packed 21 B/ray gather buffers of the 8 bands unpack to exactly that image."""
    H = W = 2048
    world = 8
    dec = gu.gpu_decoder("B")
    K, (R, T) = synth.intrinsic(H, W), synth.front_camera()
    lat, R, T = synth.make_latent().cuda(), R.cuda(), T.cuda()
    full = pkg.SDFRenderer(dec, K, img_hw=(H, W), engine="tc").render(lat, R, T, ray_marching_type=kind, no_grad=True)
    assert 0.15 < float(full[2].float().mean()) < 0.35
    bufs = []
    for r in range(world):
        sh = par.ShardedSDFRenderer(dec, K, (H, W), rank=r, world_size=world, engine="tc")
        rows = torch.tensor([y for y in range(H) if (y // 4) % world == r], device="cuda")
        band = sh.render(lat, R, T, ray_marching_type=kind, no_grad=True)
        for a, b in zip(band, full):
            assert torch.equal(a, b[rows]), (kind, r)
        bufs.append(par.pack_band(band, (H, W), world, stat=sh.local._last_counts))
        del sh
    assert bufs[0].numel() == 21 * (H // world) * W + 16
    outs, stats, _ = par.unpack_bands(torch.stack(bufs), (H, W), world)
    for a, b in zip(outs, full):
        assert torch.equal(a, b) and a.dtype == b.dtype
    assert int(stats[:, 0].sum()) == H * W      # every ray meets the unit sphere with this camera


def test_sharded_default_march_and_empty_band():
    """ADVICE r1: ShardedSDFRenderer.render with its default march (pyramid_recursive, as the reference) works on a band;
    a band without any live ray does not raise on its own (the other ranks would hang in the all-gather): the test is
    taken over the gathered statistics, on every rank alike."""
    H, W = 64, 48
    dec = gu.gpu_decoder("B")
    K, (R, T) = synth.intrinsic(H, W), synth.lookat_camera(30.0, 20.0, 2.0)
    lat, R, T = synth.make_latent().cuda(), R.cuda(), T.cuda()
    full = pkg.SDFRenderer(dec, K, img_hw=(H, W)).render(lat, R, T, no_grad=True)        # default: pyramid_recursive
    bufs = []
    for r in range(2):
        sh = par.ShardedSDFRenderer(dec, K, (H, W), rank=r, world_size=2)
        bufs.append(par.pack_band(sh.render(lat, R, T, no_grad=True), (H, W), 2, stat=sh.local._last_counts))
    outs, stats, _ = par.unpack_bands(torch.stack(bufs), (H, W), 2)
    for a, b in zip(outs, full):
        assert torch.equal(a, b)
    one = par.ShardedSDFRenderer(dec, K, (H, W), rank=0, world_size=1)
    o, _ = one.gather(one.render(lat, R, T, no_grad=True))
    for a, b in zip(o, full):
        assert torch.equal(a, b)
    # camera looking away: no ray meets the unit sphere -> the local render returns, gather() raises
    T_away = torch.tensor([50.0, 0.0, 1.6]).cuda()
    band = one.render(lat, torch.eye(3).cuda(), T_away, ray_marching_type="recursive", no_grad=True)
    with pytest.raises(ValueError):
        one.gather(band)
