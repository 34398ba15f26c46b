"""Seeded test configurations shared by oracle/make_golden.py, the CPU tests and the GPU parity tests."""
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
pkg = importlib.import_module("dist-renderer_b200")
synth = importlib.import_module("dist-renderer_b200.synth")

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

# The fp32 oracles' last bits depend on how many threads split their CPU GEMMs, and a march that starts inside the
# shape turns such bits into visible differences.  The fixtures were written with this many threads; the tests and
# oracle/make_golden.py use the same count on any host, whatever its number of cores.
CPU_THREADS = 8
torch.set_num_threads(CPU_THREADS)

# name -> recipe.  cam: ('front', dist) or ('lookat', az, el, dist, focal_scale)
CASES = {
    "c1_recursive_64": dict(decoder="B", hw=(64, 64), cam=("front", 1.6), march_step=50, buffer_size=5,
                            kind="recursive"),
    "c1_decoderA_64": dict(decoder="A", hw=(64, 64), cam=("front", 1.6), march_step=50, buffer_size=5,
                           kind="recursive"),
    "trivial_40": dict(decoder="B", hw=(40, 40), cam=("front", 1.6), march_step=50, buffer_size=5, kind="trivial"),
    "pyramid_64": dict(decoder="B", hw=(64, 64), cam=("front", 1.6), march_step=50, buffer_size=5,
                       kind="pyramid_recursive"),
    "c3_lookat_56": dict(decoder="B", hw=(56, 56), cam=("lookat", 40.0, 25.0, 2.5, 1.2 * 2.5 / 1.6),
                         march_step=100, buffer_size=3, kind="recursive"),
    "ragged_37x53": dict(decoder="B", hw=(37, 53), cam=("lookat", 200.0, -30.0, 1.9, 1.0), march_step=30,
                         buffer_size=5, kind="recursive"),
    "inside_32": dict(decoder="B", hw=(32, 32), cam=("front", 0.8), march_step=40, buffer_size=5, kind="recursive"),
    "pyramid_ragged_37x53": dict(decoder="B", hw=(37, 53), cam=("lookat", 120.0, 20.0, 2.2, 1.3), march_step=50,
                                 buffer_size=3, kind="pyramid_recursive"),
    "pyramid_inside_30": dict(decoder="B", hw=(30, 30), cam=("front", 0.85), march_step=40, buffer_size=5,
                              kind="pyramid_recursive"),
    # every ray leaves the unit sphere within fewer than buffer_size steps: the early-break padding of
    # renderer.py:562-567 (7 steps < 8; pyramid: 2 full-resolution steps < 5, copies compete with the coarse samples)
    "earlybreak_recursive_16": dict(decoder="B", hw=(16, 16), cam=("offset", 0.975, 1.6, 8.0), march_step=50,
                                    buffer_size=8, kind="recursive"),
    "earlybreak_pyramid_16": dict(decoder="B", hw=(16, 16), cam=("offset", 0.9, 1.6, 8.0), march_step=50,
                                  buffer_size=5, kind="pyramid_recursive"),
}

# BASELINE.json configurations at their own sizes (fixtures written by oracle/make_golden.py --big from the real
# reference; minutes of CPU each, so the CPU suite only checks their metadata and the GPU suite compares against them)
_RING = ("lookat", 45.0, 25.0, 2.5, 1.2 * 2.5 / 1.6)
BIG_CASES = {
    # config 2 / the bench workload: 512x512, 50 steps, buffer 5
    "c2_512_recursive": dict(decoder="B", hw=(512, 512), cam=("front", 1.6), march_step=50, buffer_size=5,
                             kind="recursive"),
    # (the reference's pyramid march at 512x512 needs more than the 62 GB of this container on CPU -- lists of all
    #  three levels are kept with their autograd graphs; the pyramid is pinned at config 3's size below)
    # config 3: run_single_shape.py:116,152-155 renderer settings at 224x224
    "c3_224_recursive": dict(decoder="B", hw=(224, 224), cam=("lookat", 40.0, 25.0, 2.5, 1.2 * 2.5 / 1.6),
                             march_step=100, buffer_size=3, kind="recursive"),
    "c3_224_pyramid": dict(decoder="B", hw=(224, 224), cam=("lookat", 40.0, 25.0, 2.5, 1.2 * 2.5 / 1.6),
                           march_step=100, buffer_size=3, kind="pyramid_recursive"),
    # config 4: one 256x256 view of the PMO ring, run_multi_pmodata.py:92 renderer settings
    "c4_256_ring": dict(decoder="B", hw=(256, 256), cam=_RING, march_step=100, buffer_size=1, kind="recursive"),
}

# one small case per gradient flag of render() (renderer.py:943-957) + the silhouette pair of render_depth
_FLAG_BASE = dict(decoder="B", hw=(48, 48), cam=("lookat", 60.0, 20.0, 2.0, 1.5), march_step=50, buffer_size=5,
                  kind="recursive")
FLAG_CASES = {
    "flag_no_grad_depth": dict(_FLAG_BASE, flags=dict(no_grad_depth=True)),
    "flag_no_grad_mask": dict(_FLAG_BASE, flags=dict(no_grad_mask=True)),
    "flag_no_grad_camera": dict(_FLAG_BASE, flags=dict(no_grad_camera=True)),
    "flag_no_grad_normal": dict(_FLAG_BASE, flags=dict(no_grad_normal=True)),
    "flag_unnormalized_normal": dict(_FLAG_BASE, flags=dict(normalize_normal=False)),
    "flag_pyramid_no_grad_camera": dict(_FLAG_BASE, kind="pyramid_recursive", flags=dict(no_grad_camera=True)),
}

_DEC = {}


def decoder(kind):
    if kind not in _DEC:
        _DEC[kind] = synth.make_decoder(kind)
    return _DEC[kind]


def camera(spec, hw):
    H, W = hw
    if spec[0] == "front":
        R, T = synth.front_camera(spec[1])
        K = synth.intrinsic(H, W)
    elif spec[0] == "offset":      # front camera shifted sideways: every ray passes at about |tx| from the origin
        _, tx, dist, fs = spec
        R, T = synth.front_camera(dist)
        T = T + torch.tensor([tx, 0.0, 0.0])
        K = synth.intrinsic(H, W, focal_scale=fs)
    else:
        _, az, el, dist, fs = spec
        R, T = synth.lookat_camera(az, el, dist)
        K = synth.intrinsic(H, W, focal_scale=fs)
    return K, R, T


LOSS_W = torch.tensor([0.3, -0.2, 0.5])


def scalar_loss(out):
    """A fixed scalar of render()'s outputs used to compare gradients: depth on the mask, min_sdf, normal."""
    depth, normal, mask, min_sdf = out
    m = mask.bool()
    return depth[m].sum() + 3.0 * min_sdf.sum() + (normal * LOSS_W.to(normal)).sum()


def weights_checksum(dec):
    with torch.no_grad():
        return float(sum(p.double().abs().sum() for p in dec.state_dict().values()))


def color_case():
    """next-3: SDFRenderer_color on a 24x24 front view, 8-d colour code, one point light with energy 0.8."""
    hw = (24, 24)
    K, R, T = camera(("front", 1.6), hw)
    g = torch.Generator().manual_seed(13)
    color_code = 0.1 * torch.randn(1, 8, generator=g)
    return hw, K, R, T, color_code, torch.tensor([[0.5, 1.0, -3.0]]), torch.tensor([0.8])


def color_lighting(lights, energies):
    """The lighting arguments of SDFRenderer_color.render compared with the reference: none, locations, both."""
    return [dict(), dict(lighting_locations=lights), dict(lighting_locations=lights, lighting_energies=energies)]


def loss_case():
    """The single-view loss (loss_single.py:7-57) on a 40x40 view; the renderer runs a 60-step march with buffer 3."""
    hw = (40, 40)
    return (hw, synth.intrinsic(*hw)) + synth.lookat_camera(30.0, 20.0, 1.8)


# depth maps fed to depth2normal (renderer.py:972-975), degenerate sizes included
D2N_SHAPES = [(7, 9), (40, 33), (3, 3), (2, 5), (1, 1)]

SMALL_SPEC = dict(dims=[64] * 8, dropout=list(range(8)), dropout_prob=0.2, norm_layers=list(range(8)), latent_in=[4],
                  xyz_in_all=False, use_tanh=False, latent_dropout=False, weight_norm=True)


def write_experiment(root, make_decoder):
    """An experiment directory in the upstream DeepSDF layout: specs.json, an SDF checkpoint saved from a DataParallel
    wrapper (keys prefixed `module.`) and a colour checkpoint saved without the prefix (decoder_utils.py:33-41).
    Returns the colour experiment's directory."""
    import json
    json.dump({"NetworkArch": "deep_sdf_decoder", "CodeLength": 16, "NetworkSpecs": SMALL_SPEC},
              open(os.path.join(root, "specs.json"), "w"))
    col = os.path.join(root, "color")
    os.makedirs(os.path.join(root, "ModelParameters"))
    os.makedirs(os.path.join(col, "ModelParameters"))
    torch.manual_seed(0)
    sdf = torch.nn.DataParallel(make_decoder(16, **SMALL_SPEC))
    torch.save({"epoch": 1, "model_state_dict": sdf.state_dict()}, os.path.join(root, "ModelParameters", "latest.pth"))
    cspec = dict(SMALL_SPEC, dims=[64, 64, 64, 72, 64, 64, 64, 64])
    torch.save({"epoch": 1, "model_state_dict": make_decoder(24, last_dim=3, **cspec).state_dict()},
               os.path.join(col, "ModelParameters", "latest.pth"))
    return col


def warp_case():
    """Two views 15 degrees apart on the ring + two seeded random images (config 4's origin: render_warp)."""
    H = W = 40
    K = synth.intrinsic(H, W, 1.2 * 2.5 / 1.6)
    v1, v2 = synth.lookat_camera(20.0, 25.0, 2.5), synth.lookat_camera(35.0, 25.0, 2.5)
    g = torch.Generator().manual_seed(9)
    img1, img2 = torch.rand(H, W, 3, generator=g), torch.rand(H, W, 3, generator=g)
    return (H, W), K, v1, v2, img1, img2
