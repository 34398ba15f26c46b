"""CPU: pin the oracles (oracle/*.py) against golden fixtures that hold outputs of the real reference
(tests/golden, written by oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

import cases
from oracle.sdf_oracle import OracleSDFRenderer, decode_sdf, decode_sdf_gradient


def _rel(a, b):
    a, b = torch.as_tensor(a, dtype=torch.float64), torch.as_tensor(b, dtype=torch.float64)
    return float((a - b).norm() / (b.norm() + 1e-300))


def _run_oracle(cs, dtype=torch.float32, flags=None):
    flags = flags or {}
    dec = cases.decoder(cs["decoder"])
    if dtype == torch.float64:
        import copy
        dec = copy.deepcopy(dec).double()
    K, R, T = cases.camera(cs["cam"], cs["hw"])
    ren = OracleSDFRenderer(dec, K, img_hw=cs["hw"], march_step=cs["march_step"], buffer_size=cs["buffer_size"],
                            dtype=dtype)
    lat = cases.synth.make_latent().to(dtype).requires_grad_(True)
    Rg, Tg = R.to(dtype).requires_grad_(True), T.to(dtype).requires_grad_(True)
    out = ren.render(lat, Rg, Tg, ray_marching_type=cs["kind"], **flags)
    cases.scalar_loss(out).backward()
    return out, tuple(t.grad if t.grad is not None else torch.zeros_like(t) for t in (lat, Rg, Tg))


@pytest.mark.parametrize("name", sorted(cases.CASES))
def test_oracle_matches_golden(name):
    """Golden = outputs of the unmodified reference.  Same torch build, same ops -> expect (near) bit equality."""
    cs = cases.CASES[name]
    gold = np.load(os.path.join(cases.GOLDEN_DIR, name + ".npz"))
    assert abs(cases.weights_checksum(cases.decoder(cs["decoder"])) - float(gold["weights_checksum"])) < 1e-6
    out, grads = _run_oracle(cs)
    assert int((out[2].numpy() != gold["mask"]).sum()) == 0
    m = gold["mask"].astype(bool)
    if m.any():
        assert _rel(out[0].detach().numpy()[m], gold["depth"][m]) < 1e-6
        assert _rel(out[1].detach().numpy(), gold["normal"]) < 1e-5
    assert _rel(out[3].detach().numpy(), gold["min_sdf"]) < 1e-6
    for g, key in zip(grads, ("g_latent", "g_R", "g_T")):
        assert _rel(g.numpy(), gold[key]) < 1e-4, key


@pytest.mark.parametrize("name", sorted(cases.FLAG_CASES))
def test_oracle_matches_flag_golden(name):
    """One fixture per gradient flag of the reference's render() (renderer.py:943-957): which of d latent / dR / dT
    survive each flag -- including the reference's quirk that the trivial march (and with it the coarse levels of the
    pyramid) ignores no_grad_camera (renderer.py:481-484 never detaches its points)."""
    cs = cases.FLAG_CASES[name]
    gold = np.load(os.path.join(cases.GOLDEN_DIR, name + ".npz"))
    out, grads = _run_oracle(cs, flags=cs["flags"])
    assert int((out[2].numpy() != gold["mask"]).sum()) == 0
    m = gold["mask"].astype(bool)
    assert _rel(out[0].detach().numpy()[m], gold["depth"][m]) < 1e-6
    assert _rel(out[1].detach().numpy(), gold["normal"]) < 1e-5
    assert _rel(out[3].detach().numpy(), gold["min_sdf"]) < 1e-6
    for g, key in zip(grads, ("g_latent", "g_R", "g_T")):
        ref = gold[key]
        if float(np.abs(ref).max()) < 1e-6:
            assert float(g.abs().max()) < 1e-6, key
        else:
            assert _rel(g.numpy(), ref) < 1e-4, key


@pytest.mark.parametrize("name", ["earlybreak_recursive_16", "earlybreak_pyramid_16"])
def test_oracle_earlybreak_padding_render_depth(name):
    """renderer.py:562-567: when every ray finishes in fewer than buffer_size steps the lists are padded with copies of
    the last step; visible in render_depth's raw Zdepth and in the gradient through all buffer_size samples."""
    cs = cases.CASES[name]
    gold = np.load(os.path.join(cases.GOLDEN_DIR, name + ".npz"))
    K, R, T = cases.camera(cs["cam"], cs["hw"])
    ren = OracleSDFRenderer(cases.decoder(cs["decoder"]), K, img_hw=cs["hw"], march_step=cs["march_step"],
                            buffer_size=cs["buffer_size"])
    lat = cases.synth.make_latent().requires_grad_(True)
    Rg, Tg = R.clone().requires_grad_(True), T.clone().requires_grad_(True)
    Zd, _, _ = ren.render_depth(lat, Rg, Tg, ray_marching_type=cs["kind"])
    Zd[Zd < 1e10].sum().backward()
    assert _rel(Zd.detach().numpy(), gold["rd_Zdepth"]) < 1e-6
    for g, key in zip((lat.grad, Rg.grad, Tg.grad), ("rd_g_latent", "rd_g_R", "rd_g_T")):
        assert _rel(g.numpy(), gold[key]) < 1e-4, key


def _golden(name):
    return np.load(os.path.join(cases.GOLDEN_DIR, name + ".npz"))


def test_loss_oracle_matches_live_reference():
    """oracle/loss_oracle.py == the reference's compute_all_loss (loss_single.py:7-57) on the reference's renderer
    (tests/golden/loss_40.npz, with the ground-truth maps it was given): every term of the loss pack, the weighted total
    and its gradient w.r.t. the shape code."""
    from oracle import loss_oracle
    gold = _golden("loss_40")
    hw, K, R, T = cases.loss_case()
    ora = OracleSDFRenderer(cases.decoder("B"), K, img_hw=hw, march_step=60, buffer_size=3)
    gt_pack = {k: torch.from_numpy(gold["gt_" + k]) for k in ("depth", "normal", "silhouette")}
    l_o = cases.synth.make_latent().requires_grad_(True)
    pack_o = loss_oracle.compute_all_loss(ora, l_o, torch.cat([R, T[:, None]], 1), gt_pack, ray_marching_type='recursive')
    loss_oracle.total(pack_o).backward()
    for k in ("mask_gt", "mask_out", "depth", "normal", "l2reg"):
        ref = float(gold["pack_" + k])
        assert abs(float(pack_o[k]) - ref) <= 1e-6 * max(1.0, abs(ref)), k
    assert float(gold["pack_depth"]) > 0 and float(gold["pack_normal"]) < 0
    assert _rel(l_o.grad.numpy(), gold["g_latent"]) < 1e-5


def test_big_fixtures_present_and_consistent():
    """The BASELINE-size fixtures (cases.BIG_CASES; written by `oracle/make_golden.py --big` from the real reference)
    are too slow to re-render in the CPU suite: check they exist, match the seeded decoder and carry their fp64 floor.
    Above 256x256 pixels a fixture holds the maps at a sample of distinct pixels (`pix`, flat indices) and the mask whole."""
    for name, cs in cases.BIG_CASES.items():
        gold = np.load(os.path.join(cases.GOLDEN_DIR, "big_" + name + ".npz"))
        assert abs(cases.weights_checksum(cases.decoder(cs["decoder"])) - float(gold["weights_checksum"])) < 1e-6
        shape = cs["hw"]
        if cs["hw"][0] * cs["hw"][1] > 256 * 256:
            pix = gold["pix"]
            assert np.all(np.diff(pix) > 0) and 0 <= pix[0] and pix[-1] < cs["hw"][0] * cs["hw"][1]
            shape = pix.shape
        assert gold["depth"].shape == shape and gold["normal"].shape == shape + (3,) and gold["min_sdf"].shape == shape
        assert gold["mask"].shape == cs["hw"] and gold["mask"].dtype == np.uint8 and 0.05 < gold["mask"].mean() < 0.6
        floor = dict(zip(gold["floor_keys"].tolist(), gold["floor_vals"].tolist()))
        assert floor["depth"] < 1e-5 and floor["xor"] <= 0.0005 * gold["mask"].size, floor


def test_oracle_decoder_points_golden():
    gold = np.load(os.path.join(cases.GOLDEN_DIR, "decoder_points.npz"))
    dec, lat = cases.decoder("B"), cases.synth.make_latent()
    pts = torch.from_numpy(gold["points"])
    assert _rel(decode_sdf(dec, lat, pts, clamp_dist=None).detach().numpy(), gold["sdf"]) < 1e-6
    p = pts.clone().requires_grad_(True)
    assert _rel(decode_sdf_gradient(dec, lat, p).detach().numpy(), gold["grad"]) < 1e-5


@pytest.mark.parametrize("name", ["trivial_40", "inside_32"])
def test_oracle_matches_live_reference(name):
    """The reference's render() without gradients (tests/golden/nograd_*.npz)."""
    cs = cases.CASES[name]
    gold = _golden("nograd_" + name)
    a = [torch.from_numpy(gold[k]) for k in ("depth", "normal", "mask", "min_sdf")]
    b, _ = _run_oracle(cs)
    assert int((a[2] != b[2]).sum()) == 0
    for i in (0, 1, 3):
        assert _rel(b[i].detach(), a[i]) < 1e-6


def test_depth2normal_matches_live_reference():
    """use_depth2normal (renderer.py:972-975): the oracle's restatement and the product's host-side mirror
    (device-agnostic PyTorch, so checked here on CPU) against the reference's own function (its outputs on the same
    seeded maps in tests/golden/depth2normal.npz), bit for bit, including the in-place zeroing of the background of the
    depth map; then the whole render() branch, oracle vs reference."""
    import importlib
    from oracle.sdf_oracle import depth2normal as d2n_oracle
    gold = _golden("depth2normal")
    d2n_prod = importlib.import_module("dist-renderer_b200.render_utils").depth2normal
    g = torch.Generator().manual_seed(3)
    for i, (h, w) in enumerate(cases.D2N_SHAPES):
        d = torch.rand(h, w, generator=g) * 2 + 0.5
        d[torch.rand(h, w, generator=g) < 0.3] = 1e11
        d[0, 0] = 0.0
        fx, fy = np.float32(57.6), np.float32(50.0)
        da, db, dc = torch.from_numpy(gold["depth_%d" % i]), d.clone(), d.clone()
        a, b, c = torch.from_numpy(gold["normal_%d" % i]), d2n_oracle(db, fx, fy), d2n_prod(dc, fx, fy)
        assert torch.equal(a, b) and torch.equal(a, c)
        assert torch.equal(da, db) and torch.equal(da, dc) and float(da[0, 0]) == 0.0
    # gradients w.r.t. the depth agree (the product forms the differences before scattering: last-bit differences)
    d = torch.rand(12, 12, generator=g) + 0.5
    d[2:4, 3] = 1e11
    wgt = torch.randn(12, 12, 3, generator=g)
    grads = [torch.from_numpy(gold["grad"])]
    for fn in (d2n_oracle, d2n_prod):
        x = d.clone().requires_grad_(True)
        (fn(x * 1.0, np.float32(30.0)) * wgt).sum().backward()
        grads.append(x.grad)
    assert torch.equal(grads[0], grads[1]) and _rel(grads[2], grads[0]) < 1e-6
    # the render() branch
    cs = cases.CASES["trivial_40"]
    K, R, T = cases.camera(cs["cam"], cs["hw"])
    kw = dict(img_hw=cs["hw"], march_step=cs["march_step"], buffer_size=cs["buffer_size"], use_depth2normal=True)
    a = [torch.from_numpy(gold["render_" + k]) for k in ("depth", "normal", "mask", "min_sdf")]
    b = OracleSDFRenderer(cases.decoder(cs["decoder"]), K, **kw).render(cases.synth.make_latent(), R, T,
                                                                         ray_marching_type="recursive", no_grad=True)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert float(a[0].min()) == 0.0 and float(a[0].max()) < 1e5      # background of the returned depth is 0, not 1e11


def test_load_decoder_roundtrip(tmp_path):
    """load_decoder (decoder_utils.py:7-51): SDF and colour decoders, DataParallel wrapper by default."""
    col = cases.write_experiment(str(tmp_path), cases.pkg.Decoder)
    wrapped = cases.pkg.load_decoder(str(tmp_path), "latest")
    assert isinstance(wrapped, torch.nn.DataParallel) and wrapped.module.latent_size == 16
    bare = cases.pkg.load_decoder(str(tmp_path), "latest", parallel=False)
    x = torch.randn(9, 19)
    # DataParallel moves the module to cuda:0 where a GPU is present: compared on the host
    assert torch.equal(wrapped.module.eval().cpu().inference(x), bare.eval().inference(x))
    colour = cases.pkg.load_decoder(str(tmp_path), "latest", color_size=8, experiment_directory_color=col).module.eval().cpu()
    assert colour.latent_size == 24 and colour.lin3.weight_v.shape[0] == 72 - 27 and colour.lin8.out_features == 3
    rgb = colour.inference(torch.cat([torch.randn(1, 16).expand(70, -1), torch.randn(1, 8).expand(70, -1), torch.randn(70, 3)], 1))
    assert rgb.shape == (70, 3) and float(rgb.abs().max()) <= 1.0
    with pytest.raises(ValueError):     # decode_color runs on the CUDA engines only (no CPU path in the product)
        cases.pkg.decode_color(colour, torch.randn(1, 8), torch.randn(1, 16), torch.randn(70, 3))
    with pytest.raises(Exception):
        cases.pkg.load_decoder(str(tmp_path / "nowhere"))


def test_load_decoder_and_decode_color_match_live_reference(tmp_path):
    """The reference's load_decoder and decode_color on the same experiment (its outputs and weight checksums in
    tests/golden/load_decoder.npz; the reference's Decoder writes the same weights as the product's)."""
    gold = _golden("load_decoder")
    col = cases.write_experiment(str(tmp_path), cases.pkg.Decoder)
    b = cases.pkg.load_decoder(str(tmp_path), "latest").module.eval().cpu()
    assert cases.weights_checksum(b) == float(gold["sdf_checksum"])
    x = torch.from_numpy(gold["x"])
    assert torch.equal(torch.from_numpy(gold["sdf"]), b.inference(x))
    bc = cases.pkg.load_decoder(str(tmp_path), "latest", color_size=8, experiment_directory_color=col).module.eval().cpu()
    assert cases.weights_checksum(bc) == float(gold["color_checksum"])
    pts, sc, cc = (torch.from_numpy(gold[k]) for k in ("pts", "shape_code", "color_code"))
    # the reference's decode_color rows are [shape code | colour code | xyz] (decoder_utils.py:103): same module outputs
    rows = torch.cat([sc.expand(70, -1), cc.expand(70, -1), pts], 1)
    assert _rel(torch.from_numpy(gold["rgb"]), bc.inference(rows).detach()) < 1e-6   # (chunked GEMMs)


def _color_setup():
    from oracle.color_oracle import OracleColorRenderer
    hw, K, R, T, cc, lights, energies = cases.color_case()
    col = cases.synth.make_color_decoder()
    ora = OracleColorRenderer(cases.decoder("B"), col, K, img_hw=hw)
    return ora, col, (hw, K, R, T, cc, lights, energies)


def test_color_oracle_matches_golden():
    """next-3: oracle/color_oracle.py vs the reference's SDFRenderer_color.render outputs in tests/golden/color_24.npz."""
    import numpy as np
    ora, col, (hw, K, R, T, cc, lights, energies) = _color_setup()
    gold = np.load(os.path.join(cases.GOLDEN_DIR, "color_24.npz"))
    assert abs(cases.weights_checksum(col) - float(gold["weights_checksum"])) < 1e-6 * float(gold["weights_checksum"])
    lat, ccg = cases.synth.make_latent().requires_grad_(True), cc.clone().requires_grad_(True)
    out = ora.render(ccg, lat, R, T, lighting_locations=lights, lighting_energies=energies)
    (out[2].sum() + out[0][out[3].bool()].sum()).backward()
    assert int((out[3].numpy() != gold["mask"]).sum()) == 0
    for i, key in ((0, "depth"), (1, "normal"), (2, "color"), (4, "min_sdf")):
        assert _rel(out[i].detach(), torch.from_numpy(gold[key])) < 1e-6, key
    assert _rel(lat.grad, torch.from_numpy(gold["g_latent"])) < 1e-5
    assert _rel(ccg.grad, torch.from_numpy(gold["g_color"])) < 1e-5
    plain = ora.render(cc, cases.synth.make_latent(), R, T, no_grad=True)
    assert _rel(plain[2], torch.from_numpy(gold["color_unlit"])) < 1e-6


def test_color_oracle_matches_live_reference():
    """Bit-for-bit against renderer_rgb.py (its outputs in tests/golden/color_lighting_24.npz): outputs under each
    lighting argument, and gradients w.r.t. both codes."""
    gold = _golden("color_lighting_24")
    ora, col, (hw, K, R, T, cc, lights, energies) = _color_setup()
    lat = cases.synth.make_latent()
    for i, kw in enumerate(cases.color_lighting(lights, energies)):
        b = ora.render(cc, lat, R, T, no_grad=True, **kw)
        assert all(torch.equal(torch.from_numpy(gold["out_%d_%d" % (i, j)]), y) for j, y in enumerate(b))
    l, c = lat.clone().requires_grad_(True), cc.clone().requires_grad_(True)
    o = ora.render(c, l, R, T, lighting_locations=lights)
    (o[2].sum() + o[0][o[3].bool()].sum()).backward()
    assert torch.equal(torch.from_numpy(gold["g_latent"]), l.grad) and torch.equal(torch.from_numpy(gold["g_color"]), c.grad)


def test_deepsdf_sampler_host_logic_matches_live_reference(monkeypatch):
    """SDFRenderer_deepsdf.get_samples / get_freespace_samples (renderer_deepsdf.py:14-65).  The product methods are
    device-agnostic host code around decode_sdf; here they run on CPU -- on a renderer object whose constructor (which
    insists on a CUDA decoder) is bypassed and whose decoder calls are routed to the oracle's decode_sdf -- against the
    reference class's outputs on the same depth and normal maps (tests/golden/deepsdf_samples_24.npz), bit for bit,
    including the random draws under a common seed."""
    import importlib
    from oracle.sdf_oracle import decode_sdf as oracle_decode
    gold = _golden("deepsdf_samples_24")
    mod = importlib.import_module("dist-renderer_b200.renderer_deepsdf")
    monkeypatch.setattr(mod.functional, "decode_sdf",
                        lambda dec, lat, pts, clamp_dist=0.1, **kw: oracle_decode(dec, lat, pts, clamp_dist=clamp_dist))
    hw = (24, 24)
    K, R, T = cases.camera(("front", 1.6), hw)
    dec = cases.decoder("B")
    lat = cases.synth.make_latent()
    depth, normal = torch.from_numpy(gold["depth"]), torch.from_numpy(gold["normal"])
    RT = torch.cat([R, T[:, None]], 1)
    prod = object.__new__(mod.SDFRenderer_deepsdf)            # no CUDA here: set what the camera helpers read
    prod.decoder, prod.device, prod.img_hw, prod.rows, prod.Pv = dec, torch.device("cpu"), hw, (0, 1, hw[0], 1), hw[0] * hw[1]
    prod.K_inv = torch.from_numpy(np.linalg.inv(K)).float()
    prod.transform_matrix = torch.tensor([[1., 0., 0.], [0., 0., -1.], [0., 1., 0.]])
    prod._homo_calib = prod._calib_map = None
    a = (torch.from_numpy(gold["fixed_0"]), torch.from_numpy(gold["fixed_1"]))
    b = prod.get_samples(lat, RT, depth.clone(), normal.clone(), use_rand=False)
    assert a[0].numel() == int(((depth < 1e5) & (depth > 0)).sum()) > 50
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert float(a[0].detach().abs().max()) < 0.05 and float(a[1].detach().abs().max()) < 0.05   # near zero: the samples straddle the surface
    for fn, args, keys in (("get_samples", (depth.clone(), normal.clone()), ("random_0", "random_1")),
                           ("get_freespace_samples", (depth.clone(),), ("freespace",))):
        x = tuple(torch.from_numpy(gold[k]) for k in keys)
        torch.manual_seed(21)
        y = getattr(prod, fn)(lat, RT, *args)
        y = y if isinstance(y, tuple) else (y,)
        assert len(x) == len(y) and all(torch.equal(p, q) for p, q in zip(x, y))
    torch.manual_seed(3)
    free = prod.get_freespace_samples(lat, RT, depth.clone(), number=3)
    assert free.numel() == 3 * a[0].numel() and float(free.min()) > -0.05       # in front of the surface the sdf is positive


def test_fp64_twin_noise_floor():
    """The fp64 twin bounds how far a faithful fp32 implementation may sit from the fp32 reference."""
    cs = cases.CASES["trivial_40"]
    o32, _ = _run_oracle(cs)
    o64, _ = _run_oracle(cs, torch.float64)
    m = o32[2].bool() & o64[2].bool()
    assert int((o32[2] != o64[2]).sum()) <= 4
    assert _rel(o32[0].detach()[m], o64[0].detach()[m]) < 1e-4


def test_no_valid_depth_raises():
    """No ray meets the unit sphere: the reference dies in `init_zdepth_valid.max()` on an empty tensor
    (renderer.py:271, RuntimeError) before reaching ValueError('No valid depth.') (renderer.py:214-215)."""
    dec = cases.decoder("B")
    K = cases.synth.intrinsic(8, 8)
    ren = OracleSDFRenderer(dec, K, img_hw=(8, 8))
    R, T = cases.synth.front_camera(50.0)      # unit sphere covers < 1 pixel and no pixel centre hits it
    K[0, 2] += 400.0                            # shift principal point so every ray misses
    ren = OracleSDFRenderer(dec, K, img_hw=(8, 8))
    with pytest.raises((ValueError, RuntimeError)):
        ren.render_depth(cases.synth.make_latent(), R, T, no_grad=True)


def test_warp_oracle_matches_golden():
    """oracle/warp_oracle.py vs the reference's render_warp outputs stored in tests/golden/warp_40.npz."""
    from oracle.warp_oracle import OracleWarpRenderer
    gold = np.load(os.path.join(cases.GOLDEN_DIR, "warp_40.npz"))
    hw, K, (R1, T1), (R2, T2), img1, img2 = cases.warp_case()
    ow = OracleWarpRenderer(cases.decoder("B"), K, img_hw=hw)
    lat = cases.synth.make_latent().requires_grad_(True)
    out = ow.render_warp(lat, R1, T1, R2, T2, img1, img2)
    out[0].backward()
    assert abs(float(out[0]) - float(gold["loss"])) < 1e-6
    assert _rel(lat.grad.numpy(), gold["g_latent"]) < 1e-4
    assert int((out[1].numpy() != gold["mask1"]).sum()) == 0 and int((out[2].numpy() != gold["mask2"]).sum()) == 0
    assert _rel(out[6].detach().numpy(), gold["depth1"]) < 1e-6


def test_warp_oracle_matches_live_reference():
    """The reference's render_warp loss and first-view normals (tests/golden/warp_40.npz) at the tight bar."""
    from oracle.warp_oracle import OracleWarpRenderer
    gold = _golden("warp_40")
    hw, K, (R1, T1), (R2, T2), img1, img2 = cases.warp_case()
    b = OracleWarpRenderer(cases.decoder("B"), K, img_hw=hw).render_warp(cases.synth.make_latent(), R1, T1, R2, T2, img1, img2)
    assert abs(float(gold["loss"]) - float(b[0])) < 1e-7
    assert _rel(b[5].detach(), torch.from_numpy(gold["normal1"])) < 1e-6


def test_grid_oracle_matches_live_reference():
    """oracle/grid_oracle.py vs the reference's create_mesh.py sampling functions (next-2): the sample coordinates and
    the sparse-evaluated grid, bit for bit (sha256 of the reference's arrays in tests/golden/grid_64.npz)."""
    import hashlib
    from oracle import grid_oracle
    gold = _golden("grid_64")
    digest = lambda t: hashlib.sha256(np.ascontiguousarray(t.numpy()).tobytes()).hexdigest()
    N = 64          # 1.5 coarse voxels = 0.097 < the 0.1 clamp: the near/far classification becomes selective
    vs = 2.0 / (N - 1)
    assert digest(grid_oracle.get_samples(N, [-1, -1, -1], vs, True)) == str(gold["coords_sha256"])
    og, n = grid_oracle.grid_speedup(cases.decoder("B"), cases.synth.make_latent(), N)
    assert digest(og) == str(gold["grid_sha256"]) and 0 < n < N ** 3
