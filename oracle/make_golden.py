"""TEST INFRASTRUCTURE ONLY -- writes tests/golden/*.npz from the REAL reference (via oracle/ref_shim.py).

Run where the reference tree is (DIST_REFERENCE_ROOT): python oracle/make_golden.py            (small cases)
                                                       python oracle/make_golden.py --flags    (gradient flags)
                                                       python oracle/make_golden.py --big      (BASELINE sizes; ~20 min)
                                                       python oracle/make_golden.py --chamfer  (eval_func.py outputs)
                                                       python oracle/make_golden.py --reference (oracle pins)
Each fixture holds the outputs of the unmodified reference `SDFRenderer.render` (depth, normal, mask, min_sdf),
the gradients of tests/cases.scalar_loss w.r.t. latent / R / T, and a checksum of the seeded decoder weights
the recipe regenerates.  `decoder_points.npz` pins decode_sdf / decode_sdf_gradient on random points.
"""
import hashlib
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
warnings.filterwarnings("ignore")

from oracle import ref_shim  # noqa: E402
import cases  # noqa: E402


def ref_decoder(dec):
    _, _, RefDecoder = ref_shim.load()
    ref = RefDecoder(dec.latent_size, **cases.synth.STANDARD_SPEC).eval()
    ref.load_state_dict(dec.state_dict())
    return ref


def ref_color_decoder(col):
    _, _, RefDecoder = ref_shim.load()
    ref_col = RefDecoder(col.latent_size, last_dim=3, **dict(cases.synth.STANDARD_SPEC, dims=list(col.dims[1:-1]))).eval()
    ref_col.load_state_dict(col.state_dict())
    return ref_col


def color_fixture():
    """tests/golden/color_24.npz from the reference's SDFRenderer_color.render (core/sdfrenderer/renderer_rgb.py:70)."""
    Color = ref_shim.load_color()
    dec, col = cases.decoder("B"), cases.synth.make_color_decoder()
    hw, K, R, T, cc, lights, energies = cases.color_case()
    ren = Color(ref_decoder(dec), ref_color_decoder(col), K, img_hw=hw, use_gpu=False)
    lat = cases.synth.make_latent().requires_grad_(True)
    ccg = cc.clone().requires_grad_(True)
    out = ren.render(ccg, lat, R, T, lighting_locations=lights, lighting_energies=energies)
    (out[2].sum() + out[0][out[3].bool()].sum()).backward()
    plain = ren.render(cc, cases.synth.make_latent(), R, T, no_grad=True)
    np.savez_compressed(os.path.join(cases.GOLDEN_DIR, "color_24.npz"), depth=out[0].detach().numpy(),
                        normal=out[1].detach().numpy(), color=out[2].detach().numpy(), mask=out[3].numpy(),
                        min_sdf=out[4].detach().numpy(), color_unlit=plain[2].numpy(), g_latent=lat.grad.numpy(),
                        g_color=ccg.grad.numpy(), weights_checksum=cases.weights_checksum(col))
    print("color_24 hits", int(out[3].sum()), "max rgb", float(out[2].abs().max()))


def _grads(ts):
    return [t.grad.numpy() if t.grad is not None else np.zeros(tuple(t.shape), np.float32) for t in ts]


BIG_SAMPLE = 16384     # pixels kept of an image larger than 256x256 (keeps each fixture well under 1 MB)


def big_fixtures(names=None):
    """tests/golden/big_*.npz: the BASELINE.json configurations at their own sizes (cases.BIG_CASES), rendered by the
    real reference (fp32) -- outputs, gradients of cases.scalar_loss w.r.t. latent / R / T -- plus the deviation of the
    fp64 twin (oracle/sdf_oracle.py in float64, itself pinned bit for bit to the reference in fp32) from them: the noise
    floor BASELINE.md section 3 asks to be printed beside every parity number.

    Above 256x256 pixels the mask is stored whole and depth / normal / min_sdf at BIG_SAMPLE pixels drawn once with a
    fixed seed (flat indices in `pix`); the floor is then measured on those pixels too, the mask XOR on all of them."""
    import time
    import gpu_util as gu
    Rmod, _, _ = ref_shim.load()
    lat0 = cases.synth.make_latent()
    for name, cs in cases.BIG_CASES.items():
        if names and name not in names:
            continue
        t0 = time.time()
        dec = cases.decoder(cs["decoder"])
        K, R, T = cases.camera(cs["cam"], cs["hw"])
        ren = Rmod.SDFRenderer(ref_decoder(dec), K, img_hw=cs["hw"], march_step=cs["march_step"],
                               buffer_size=cs["buffer_size"], use_gpu=False)
        lat, Rg, Tg = lat0.clone().requires_grad_(True), R.clone().requires_grad_(True), T.clone().requires_grad_(True)
        out = ren.render(lat, Rg, Tg, ray_marching_type=cs["kind"])
        cases.scalar_loss(out).backward()
        ref = [o.detach() for o in out]
        gref = [torch.from_numpy(g) for g in _grads((lat, Rg, Tg))]
        t1 = time.time()
        o64, g64 = gu.run_oracle(cs, dtype=torch.float64)
        o64 = [o.float() if o.dtype == torch.float64 else o for o in o64]
        mask, maps = ref[2], {}
        if mask.numel() > 256 * 256:
            pix = np.sort(np.random.default_rng(5).choice(mask.numel(), BIG_SAMPLE, replace=False)).astype(np.int32)
            maps["pix"] = pix
            floor = gu.measure(gu.at_pixels(o64, pix), gu.at_pixels(ref, pix), [g.float() for g in g64], gref)
            floor["xor"] = int((o64[2] != mask).sum())
            ref = gu.at_pixels(ref, pix)
        else:
            floor = gu.measure(o64, ref, [g.float() for g in g64], gref)
        floor = {k: (-1.0 if v is None else float(v)) for k, v in floor.items()}
        np.savez_compressed(
            os.path.join(cases.GOLDEN_DIR, "big_" + name + ".npz"), **maps,
            depth=ref[0].numpy(), normal=ref[1].numpy(), mask=mask.numpy(), min_sdf=ref[3].numpy(),
            g_latent=gref[0].numpy(), g_R=gref[1].numpy(), g_T=gref[2].numpy(),
            floor_keys=np.array(sorted(floor)), floor_vals=np.array([floor[k] for k in sorted(floor)]),
            weights_checksum=cases.weights_checksum(dec))
        print("big_" + name, "hits", int(mask.sum()), "of", mask.numel(), "ref %.0fs fp64 %.0fs" % (t1 - t0, time.time() - t1),
              "fp64 floor:", {k: ("%.3g" % v) for k, v in floor.items()}, flush=True)


def flag_fixtures():
    """tests/golden/flag_*.npz: render() of the real reference under each gradient flag (renderer.py:943-957) with the
    gradients that survive it (zeros where autograd gives None), and silhouette_48.npz: the (valid_mask, min_sdf)
    pair of render_depth (renderer.py:878) with the gradients of min_sdf.sum()."""
    Rmod, _, _ = ref_shim.load()
    lat0 = cases.synth.make_latent()
    for name, cs in cases.FLAG_CASES.items():
        dec = cases.decoder(cs["decoder"])
        K, R, T = cases.camera(cs["cam"], cs["hw"])
        ren = Rmod.SDFRenderer(ref_decoder(dec), K, img_hw=cs["hw"], march_step=cs["march_step"],
                               buffer_size=cs["buffer_size"], use_gpu=False)
        lat, Rg, Tg = lat0.clone().requires_grad_(True), R.clone().requires_grad_(True), T.clone().requires_grad_(True)
        out = ren.render(lat, Rg, Tg, ray_marching_type=cs["kind"], **cs["flags"])
        cases.scalar_loss(out).backward()
        g = _grads((lat, Rg, Tg))
        np.savez_compressed(os.path.join(cases.GOLDEN_DIR, name + ".npz"), depth=out[0].detach().numpy(),
                            normal=out[1].detach().numpy(), mask=out[2].numpy(), min_sdf=out[3].detach().numpy(),
                            g_latent=g[0], g_R=g[1], g_T=g[2], weights_checksum=cases.weights_checksum(dec))
        print(name, "hits", int(out[2].sum()), "|g|", [float(np.abs(x).sum()) for x in g])
    cs = cases._FLAG_BASE
    dec = cases.decoder(cs["decoder"])
    K, R, T = cases.camera(cs["cam"], cs["hw"])
    ren = Rmod.SDFRenderer(ref_decoder(dec), K, img_hw=cs["hw"], march_step=cs["march_step"],
                           buffer_size=cs["buffer_size"], use_gpu=False)
    lat, Rg, Tg = lat0.clone().requires_grad_(True), R.clone().requires_grad_(True), T.clone().requires_grad_(True)
    _, vm, ms = ren.render_depth(lat, Rg, Tg, ray_marching_type=cs["kind"])
    ms.sum().backward()
    g = _grads((lat, Rg, Tg))
    np.savez_compressed(os.path.join(cases.GOLDEN_DIR, "silhouette_48.npz"), mask=vm.reshape(cs["hw"]).numpy(),
                        min_sdf=ms.detach().reshape(cs["hw"]).numpy(), g_latent=g[0], g_R=g[1], g_T=g[2],
                        weights_checksum=cases.weights_checksum(dec))
    print("silhouette_48 hits", int(vm.sum()))


def chamfer_fixture():
    """Outputs of the reference's core/evaluation/eval_func.py on the seeded point sets of tests/test_mesh_cpu.py."""
    EF = ref_shim.load_eval_func()
    rng = np.random.default_rng(7)
    a = rng.standard_normal((3000, 3)) * 0.3
    b = rng.standard_normal((2500, 3)) * 0.3 + 0.05
    np.savez_compressed(os.path.join(cases.GOLDEN_DIR, "chamfer.npz"), a=a, b=b, sq=EF.compute_chamfer_distance(a, b),
                        lin=EF.compute_chamfer_distance(a, b, use_square_dist=False),
                        sep=np.array(EF.compute_chamfer_distance_separate(a, b)))
    print("chamfer", EF.compute_chamfer_distance(a, b))


def _save(name, **arrays):
    np.savez_compressed(os.path.join(cases.GOLDEN_DIR, name + ".npz"), **arrays)
    print(name, sorted(arrays))


def _digest(t):
    """sha256 of a tensor's bytes: an exact comparison of an array too large to store."""
    return hashlib.sha256(np.ascontiguousarray(t.detach().numpy()).tobytes()).hexdigest()


def reference_fixtures():
    """What the oracle-vs-reference tests of tests/test_oracle.py compare against, computed by the reference: the loss
    pack of compute_all_loss, render() without gradients, depth2normal, load_decoder / decode_color, the colour and
    DeepSDF-sampling renderers and the mesh-grid sampling of create_mesh.py."""
    import tempfile
    from oracle import loss_oracle
    from oracle.sdf_oracle import OracleSDFRenderer
    Rmod, DU, RefDecoder = ref_shim.load()
    dec = cases.decoder("B")
    ref_dec = ref_decoder(dec)

    # compute_all_loss (loss_single.py:7-57) on the reference's renderer; ground truth rendered by the oracle
    hw, K, R, T = cases.loss_case()
    gt = OracleSDFRenderer(dec, K, img_hw=hw, march_step=60, buffer_size=3).render(
        cases.synth.make_latent(seed=2), R, T, no_grad=True)
    gt_pack = {"depth": gt[0].detach(), "normal": gt[1].detach(), "silhouette": gt[2].detach()}
    ren = Rmod.SDFRenderer(ref_dec, K, img_hw=hw, march_step=60, buffer_size=3, use_gpu=False)
    lat = cases.synth.make_latent().requires_grad_(True)
    pack, _ = ref_shim.load_loss_single()(ren, lat, torch.cat([R, T[:, None]], 1), gt_pack, ray_marching_type='recursive')
    loss_oracle.total(pack).backward()
    _save("loss_40", **{"gt_" + k: v.numpy() for k, v in gt_pack.items()},
          **{"pack_" + k: float(pack[k]) for k in ("mask_gt", "mask_out", "depth", "normal", "l2reg")},
          g_latent=lat.grad.numpy())

    # render() without gradients
    for name in ("trivial_40", "inside_32"):
        cs = cases.CASES[name]
        K, R, T = cases.camera(cs["cam"], cs["hw"])
        ren = Rmod.SDFRenderer(ref_decoder(cases.decoder(cs["decoder"])), K, img_hw=cs["hw"], march_step=cs["march_step"],
                               buffer_size=cs["buffer_size"], use_gpu=False)
        out = ren.render(cases.synth.make_latent(), R, T, ray_marching_type=cs["kind"], no_grad=True)
        _save("nograd_" + name, **{k: o.detach().numpy() for k, o in zip(("depth", "normal", "mask", "min_sdf"), out)})

    # depth2normal (renderer.py:972-975) on the seeded maps of test_depth2normal_matches_live_reference
    d2n = sys.modules["core.utils.render_utils"].depth2normal
    g = torch.Generator().manual_seed(3)
    maps = {}
    for i, (h, w) in enumerate(cases.D2N_SHAPES):
        d = torch.rand(h, w, generator=g) * 2 + 0.5
        d[torch.rand(h, w, generator=g) < 0.3] = 1e11
        d[0, 0] = 0.0
        maps["normal_%d" % i] = d2n(d, np.float32(57.6), np.float32(50.0)).detach().numpy()
        maps["depth_%d" % i] = d.numpy()           # the background zeroed in place
    d = torch.rand(12, 12, generator=g) + 0.5
    d[2:4, 3] = 1e11
    wgt = torch.randn(12, 12, 3, generator=g)
    x = d.clone().requires_grad_(True)
    (d2n(x * 1.0, np.float32(30.0)) * wgt).sum().backward()
    cs = cases.CASES["trivial_40"]
    K, R, T = cases.camera(cs["cam"], cs["hw"])
    out = Rmod.SDFRenderer(ref_dec, K, use_gpu=False, img_hw=cs["hw"], march_step=cs["march_step"],
                           buffer_size=cs["buffer_size"], use_depth2normal=True).render(
        cases.synth.make_latent(), R, T, ray_marching_type="recursive", no_grad=True)
    _save("depth2normal", **maps, grad=x.grad.numpy(),
          **{"render_" + k: o.detach().numpy() for k, o in zip(("depth", "normal", "mask", "min_sdf"), out)})

    # load_decoder / decode_color (decoder_utils.py:7-51, 94-112) on an experiment written with the reference's Decoder
    with tempfile.TemporaryDirectory() as root:
        col = cases.write_experiment(root, RefDecoder)
        a = DU.load_decoder(root, "latest").module.eval()
        ac = DU.load_decoder(root, "latest", color_size=8, experiment_directory_color=col).module.eval()
    g = torch.Generator().manual_seed(4)
    x, pts = torch.randn(50, 19, generator=g), torch.randn(70, 3, generator=g)
    sc, cc = torch.randn(1, 16, generator=g), torch.randn(1, 8, generator=g)
    _save("load_decoder", x=x.numpy(), sdf=a.inference(x).detach().numpy(), pts=pts.numpy(), shape_code=sc.numpy(),
          color_code=cc.numpy(), rgb=DU.decode_color(ac, cc, sc, pts, MAX_POINTS=32).detach().numpy(),
          sdf_checksum=cases.weights_checksum(a), color_checksum=cases.weights_checksum(ac))

    # SDFRenderer_color.render (renderer_rgb.py:70) under each lighting argument, and its gradients
    col = cases.synth.make_color_decoder()
    hw, K, R, T, cc, lights, energies = cases.color_case()
    ren = ref_shim.load_color()(ref_dec, ref_color_decoder(col), K, img_hw=hw, use_gpu=False)
    lat = cases.synth.make_latent()
    outs = {}
    for i, kw in enumerate(cases.color_lighting(lights, energies)):
        for j, o in enumerate(ren.render(cc, lat, R, T, no_grad=True, **kw)):
            outs["out_%d_%d" % (i, j)] = o.detach().numpy()
    l, c = lat.clone().requires_grad_(True), cc.clone().requires_grad_(True)
    o = ren.render(c, l, R, T, lighting_locations=lights)
    (o[2].sum() + o[0][o[3].bool()].sum()).backward()
    _save("color_lighting_24", **outs, g_latent=l.grad.numpy(), g_color=c.grad.numpy())

    # SDFRenderer_deepsdf.get_samples / get_freespace_samples (renderer_deepsdf.py:14-65) on an oracle render
    hw = (24, 24)
    K, R, T = cases.camera(("front", 1.6), hw)
    lat = cases.synth.make_latent()
    depth, normal, _, _ = OracleSDFRenderer(dec, K, img_hw=hw).render(lat, R, T, ray_marching_type="recursive", no_grad=True)
    RT = torch.cat([R, T[:, None]], 1)
    ref = ref_shim.load_deepsdf()(ref_dec, K, img_hw=hw, use_gpu=False)
    a = ref.get_samples(lat, RT, depth.clone(), normal.clone(), use_rand=False)
    torch.manual_seed(21)
    s = ref.get_samples(lat, RT, depth.clone(), normal.clone())
    torch.manual_seed(21)
    f = ref.get_freespace_samples(lat, RT, depth.clone())
    _save("deepsdf_samples_24", depth=depth.numpy(), normal=normal.numpy(), fixed_0=a[0].detach().numpy(),
          fixed_1=a[1].detach().numpy(), random_0=s[0].detach().numpy(), random_1=s[1].detach().numpy(),
          freespace=f.detach().numpy())

    # create_mesh.py's grid sampling at N = 64 (262,144 points: stored as digests)
    CM = ref_shim.load_create_mesh()
    N = 64
    vs, vsh = 2.0 / (N - 1), 2.0 / (N / 2 - 1)
    coords = CM.get_samples(N, [-1, -1, -1], vs, transform=True)[:, :3]
    sh = CM.get_samples(int(N / 2), [-1, -1, -1], vsh)
    up = CM.upsample_cubic(CM.infer_samples(ref_dec, lat, sh), int(N / 2), N)
    pos, neg, val = CM.check_valid(up, vsh)
    s = CM.get_samples(N, [-1, -1, -1], vs)
    s[pos, 3], s[neg, 3] = 0.1, -0.1
    s[val, 3] = CM.infer_samples(ref_dec, lat, s[val, :])
    _save("grid_64", coords_sha256=_digest(coords), grid_sha256=_digest(s[:, 3].reshape(N, N, N)))


def main():
    if "--chamfer" in sys.argv:
        os.makedirs(cases.GOLDEN_DIR, exist_ok=True)
        return chamfer_fixture()
    if "--reference" in sys.argv:
        os.makedirs(cases.GOLDEN_DIR, exist_ok=True)
        return reference_fixtures()
    if "--big" in sys.argv:              # minutes of CPU per case: written separately from the small fixtures
        os.makedirs(cases.GOLDEN_DIR, exist_ok=True)
        return big_fixtures([a for a in sys.argv[1:] if not a.startswith("--")])
    if "--flags" in sys.argv:
        os.makedirs(cases.GOLDEN_DIR, exist_ok=True)
        return flag_fixtures()
    if "--color-only" in sys.argv:      # adds the colour fixture without rewriting the others
        os.makedirs(cases.GOLDEN_DIR, exist_ok=True)
        return color_fixture()
    Rmod, DU, _ = ref_shim.load()
    os.makedirs(cases.GOLDEN_DIR, exist_ok=True)
    lat0 = cases.synth.make_latent()
    only = sys.argv[sys.argv.index("--only") + 1:] if "--only" in sys.argv else None   # add fixtures without rewriting the rest
    for name, cs in cases.CASES.items():
        if only is not None and name not in only:
            continue
        dec = cases.decoder(cs["decoder"])
        ref = ref_decoder(dec)
        K, R, T = cases.camera(cs["cam"], cs["hw"])
        ren = Rmod.SDFRenderer(ref, K, img_hw=cs["hw"], march_step=cs["march_step"], buffer_size=cs["buffer_size"],
                               use_gpu=False)
        lat = lat0.clone().requires_grad_(True)
        Rg, Tg = R.clone().requires_grad_(True), T.clone().requires_grad_(True)
        out = ren.render(lat, Rg, Tg, ray_marching_type=cs["kind"])
        cases.scalar_loss(out).backward()
        Zdepth, zmask, zmin = ren.render_depth(lat0, R, T, ray_marching_type=cs["kind"], no_grad=True)
        more = {}
        if name.startswith("earlybreak"):
            # no ray converges in these cases, so render() hides Zdepth: pin render_depth itself -- the raw Zdepth of the
            # sphere-hit rays and the gradients of their sum, which run through ALL buffer_size selected samples
            l2, R2, T2 = lat0.clone().requires_grad_(True), R.clone().requires_grad_(True), T.clone().requires_grad_(True)
            Zd, _, _ = ren.render_depth(l2, R2, T2, ray_marching_type=cs["kind"])
            Zd[Zd < 1e10].sum().backward()
            more = dict(rd_Zdepth=Zd.detach().numpy(), rd_g_latent=l2.grad.numpy(), rd_g_R=R2.grad.numpy(),
                        rd_g_T=T2.grad.numpy())
        np.savez_compressed(
            os.path.join(cases.GOLDEN_DIR, name + ".npz"), **more,
            depth=out[0].detach().numpy(), normal=out[1].detach().numpy(), mask=out[2].numpy(),
            min_sdf=out[3].detach().numpy(), g_latent=lat.grad.numpy(), g_R=Rg.grad.numpy(), g_T=Tg.grad.numpy(),
            Zdepth_nograd=Zdepth.numpy(), weights_checksum=cases.weights_checksum(dec))
        print(name, "hits", int(out[2].sum()), "of", out[2].numel())
    if only is not None:
        return
    # decoder-level fixture
    dec = cases.decoder("B")
    ref = ref_decoder(dec)
    g = torch.Generator().manual_seed(7)
    pts = (torch.rand(3000, 3, generator=g) - 0.5) * 1.6
    sdf = DU.decode_sdf(ref, lat0, pts, clamp_dist=None).detach()
    p = pts.clone().requires_grad_(True)
    grad = DU.decode_sdf_gradient(ref, lat0, p, clamp_dist=0.1).detach()
    np.savez_compressed(os.path.join(cases.GOLDEN_DIR, "decoder_points.npz"), points=pts.numpy(), sdf=sdf.numpy(),
                        grad=grad.numpy(), weights_checksum=cases.weights_checksum(dec))
    print("decoder_points", float(sdf.min()), float(sdf.max()))
    # two-view warp fixture (reference SDFRenderer_warp.render_warp, core/sdfrenderer/renderer_warp.py:103)
    Warp = ref_shim.load_warp()
    hw, K, (R1, T1), (R2, T2), img1, img2 = cases.warp_case()
    rw = Warp(ref, K, img_hw=hw, use_gpu=False)
    lat = lat0.clone().requires_grad_(True)
    out = rw.render_warp(lat, R1, T1, R2, T2, img1, img2)
    out[0].backward()
    np.savez_compressed(os.path.join(cases.GOLDEN_DIR, "warp_40.npz"), loss=float(out[0]), g_latent=lat.grad.numpy(),
                        mask1=out[3].numpy(), mask2=out[4].numpy(), min_sdf1=out[5].detach().numpy(),
                        normal1=out[7].detach().numpy(), depth1=out[8].detach().numpy(),
                        weights_checksum=cases.weights_checksum(dec))
    print("warp_40 loss", float(out[0]))
    color_fixture()


if __name__ == "__main__":
    main()
