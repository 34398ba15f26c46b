"""Helpers shared by the GPU parity tests."""
import copy

import numpy as np
import torch

import cases
from oracle.sdf_oracle import OracleSDFRenderer

pkg = cases.pkg


def rel(a, b):
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-300))


_GPU_DEC = {}


def gpu_decoder(kind):
    if kind not in _GPU_DEC:
        _GPU_DEC[kind] = copy.deepcopy(cases.decoder(kind)).cuda()
    return _GPU_DEC[kind]


def run_gpu(cs, engine=None, grads=True, dec=None, dec_kind=None):
    dev = torch.device("cuda")
    dec = dec if dec is not None else gpu_decoder(dec_kind or cs["decoder"])
    K, R, T = cases.camera(cs["cam"], cs["hw"])
    ren = pkg.SDFRenderer(dec, K, img_hw=cs["hw"], march_step=cs["march_step"], buffer_size=cs["buffer_size"],
                          engine=engine)
    lat = cases.synth.make_latent(dec.latent_size).to(dev).requires_grad_(grads)
    Rg, Tg = R.to(dev).requires_grad_(grads), T.to(dev).requires_grad_(grads)
    out = ren.render(lat, Rg, Tg, ray_marching_type=cs["kind"], no_grad=not grads)
    g = None
    if grads:
        cases.scalar_loss(out).backward()
        g = (lat.grad.cpu(), Rg.grad.cpu(), Tg.grad.cpu())
    return [o.detach().cpu() for o in out], g, ren


def run_oracle(cs, grads=True, dec=None, dtype=torch.float32):
    dec = dec if dec is not None else cases.decoder(cs["decoder"])
    if dtype == torch.float64:
        dec = copy.deepcopy(dec).double()
    K, R, T = cases.camera(cs["cam"], cs["hw"])
    ren = OracleSDFRenderer(dec, K, img_hw=cs["hw"], march_step=cs["march_step"], buffer_size=cs["buffer_size"],
                            dtype=dtype)
    lat = cases.synth.make_latent(dec.latent_size).to(dtype).requires_grad_(grads)
    Rg, Tg = R.to(dtype).requires_grad_(grads), T.to(dtype).requires_grad_(grads)
    out = ren.render(lat, Rg, Tg, ray_marching_type=cs["kind"], no_grad=not grads)
    g = None
    if grads:
        cases.scalar_loss(out).backward()
        g = (lat.grad, Rg.grad, Tg.grad)
    return [o.detach() for o in out], g


def at_pixels(maps, pix):
    """(depth, normal, mask, min_sdf) maps restricted to the flat pixel indices `pix` (a fixture's stored sample)."""
    idx = torch.as_tensor(pix, dtype=torch.long)
    return [m.reshape(-1, *m.shape[2:])[idx] for m in maps]


def normal_error(n_a, n_b, mask, outlier_frac=0.005, outlier_thresh=1e-3):
    """rel-L2 of the normal map on `mask` after dropping at most outlier_frac pixels whose per-pixel error exceeds
    outlier_thresh (ReLU-boundary flips: the fp32 reference vs its own fp64 twin shows the same, SURVEY.md H2).
    End to end the hit points of two faithful fp32 renders differ by ~1e-6, and the 8x512 ReLU hyperplanes are dense
    enough that a few in a thousand pixels change linear region (the fp32-vs-fp64 twin floor of SURVEY H2 is
    rel-L2 1.7e-4 *including* them), hence 0.5 % here; test_render_normal_isolated feeds identical hit points and
    holds the strict 0.1 % bar.
    Returns (rel_l2_without_outliers, n_outliers, n_allowed)."""
    a = torch.as_tensor(n_a).double().reshape(-1, 3)[mask.reshape(-1)]
    b = torch.as_tensor(n_b).double().reshape(-1, 3)[mask.reshape(-1)]
    if a.shape[0] == 0:
        return 0.0, 0, 0
    err = (a - b).norm(dim=1)
    bad = err > outlier_thresh
    allowed = max(3, int(np.ceil(outlier_frac * a.shape[0])))
    keep = ~bad
    r = float((a[keep] - b[keep]).norm() / (b[keep].norm() + 1e-300))
    return r, int(bad.sum()), allowed


def measure(out, ref, g=None, gref=None, threshold=5e-5):
    """The parity numbers of BASELINE.md section 3, without asserting: mask XOR, depth rel-L2 on the mask
    intersection, normal rel-L2 after the outlier exclusion (+ outlier count), min_sdf split into converged pixels
    (max abs) and the rest (rel-L2) plus the plain rel-L2 over all P as the gate words it, gradient rel-L2."""
    m = out[2].bool() & ref[2].bool()
    res = dict(xor=int((out[2] != ref[2]).sum()), hits=int(ref[2].sum()))
    if m.any():
        res["depth"] = rel(out[0][m], ref[0][m])
        res["normal"], res["n_out"], res["n_allowed"] = normal_error(out[1], ref[1], m)
        _, res["n_out_strict_allowed"] = None, max(3, int(np.ceil(0.001 * int(m.sum()))))
    a, b = out[3].reshape(-1).double(), ref[3].reshape(-1).double()
    conv = (a.abs() <= threshold) & (b.abs() <= threshold)
    res["min_sdf"] = rel(a[~conv], b[~conv]) if bool((~conv).any()) else 0.0
    res["min_sdf_converged_maxabs"] = float((a[conv] - b[conv]).abs().max()) if bool(conv.any()) else 0.0
    res["min_sdf_all_P"] = rel(a, b)
    if g is not None:
        for name, x, y in zip(("g_latent", "g_R", "g_T"), g, gref):
            res[name] = rel(x, y)
    return res


def compare(out, ref, g=None, gref=None, tol=1e-4, gtol=2e-3, max_xor=2, threshold=5e-5):
    """Asserts the parity bar of BASELINE.md section 3 and returns the measured numbers.

    min_sdf: a ray stops at the first sample with |sdf| < threshold (renderer.py:560), so where both renders
    converged the stored value is "some residual below the threshold" -- fp32 rounding decides whether the ray
    took one more step (e.g. 4.99e-5 stops, 5.01e-5 continues to -4.5e-5).  Those pixels are compared
    absolutely (|a-b| <= 2*threshold); everything else by rel-L2 (the plain rel-L2 over all P is reported too)."""
    res = measure(out, ref, g, gref, threshold)
    assert res["xor"] <= max_xor, res
    if "depth" in res:
        assert res["depth"] < tol, res
        assert res["normal"] < tol and res["n_out"] <= res["n_allowed"], res
    assert res["min_sdf"] < tol and res["min_sdf_converged_maxabs"] <= 2 * threshold, res
    if g is not None:
        for name in ("g_latent", "g_R", "g_T"):
            assert res[name] < gtol, res
    return res
