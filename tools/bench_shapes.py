"""Several shapes in one fused march: S shape codes at the config-3 settings (224x224, march_step 100, buffer_size 3, decoder
B, fwd+bwd with bench.loss_of), rendered as S sequential render() calls -- the per-shape loop of run_single_shape.py --
against ONE render_views() call with (S, L) codes.  The two arms alternate in the same process and are event-timed after
warm-up; the timed rounds are repeated to show the spread.  Also asserts that the two arms produce equal maps.

    python tools/bench_shapes.py [--rounds 5] [--iters 4]      (prints the table; profiles/r3_bench_shapes.txt)
"""
import argparse
import importlib
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402

pkg = importlib.import_module("dist-renderer_b200")
synth = importlib.import_module("dist-renderer_b200.synth")

HW, MARCH_STEP, BUFFER = 224, 100, 3


def gpu_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return "%s | nvidia-smi: %s" % (torch.cuda.get_device_name(0), q.splitlines()[0] if q else "?")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="1,2,4,8,16")
    ap.add_argument("--kinds", default="recursive,pyramid_recursive")
    ap.add_argument("--rounds", type=int, default=5, help="timed rounds per arm (alternating)")
    ap.add_argument("--iters", type=int, default=4, help="iterations per timed round")
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda")
    dec = synth.make_decoder("B").to(dev)
    ren = pkg.SDFRenderer(dec, synth.intrinsic(HW, HW, 1.2 * 2.5 / 1.6), img_hw=(HW, HW), march_step=MARCH_STEP,
                          buffer_size=BUFFER)
    print("# bench_shapes: S shape codes, config 3 (%dx%d, march_step %d, buffer_size %d, decoder B), fwd+bwd of "
          "bench.loss_of per shape" % (HW, HW, MARCH_STEP, BUFFER))
    print("# GPU:", gpu_line())
    print("# sequential = S render() calls (one backward each); batched = one render_views() with (S, L) codes (one "
          "backward)")
    print("# ms per shape-iteration: median [min, max] over %d rounds of %d iterations, arms alternating"
          % (args.rounds, args.iters))
    print("%-18s %3s  %-26s %-26s %9s  %s" % ("kind", "S", "sequential ms/shape", "batched ms/shape", "speed-up",
                                              "Mrays/s seq -> batched"))
    for kind in args.kinds.split(","):
        for S in [int(s) for s in args.shapes.split(",")]:
            codes = torch.cat([synth.make_latent(seed=100 + s) for s in range(S)], 0).to(dev)
            cams = [synth.lookat_camera(40.0 + 360.0 / 16 * s, 25.0, 2.5) for s in range(S)]
            Rs = torch.stack([R for R, _ in cams]).to(dev)
            Ts = torch.stack([T for _, T in cams]).to(dev)

            def sequential():
                outs = []
                for s in range(S):
                    lat = codes[s:s + 1].detach().requires_grad_(True)
                    out = ren.render(lat, Rs[s], Ts[s], ray_marching_type=kind)
                    bench.loss_of(out).backward()
                    outs.append(out)
                return outs

            def batched():
                lat = codes.detach().requires_grad_(True)
                out = ren.render_views(lat, Rs, Ts, ray_marching_type=kind)
                sum(bench.loss_of(tuple(x[s] for x in out)) for s in range(S)).backward()
                return out

            def timed(fn):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.iters):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / args.iters / S
            for _ in range(args.warmup):
                sequential()
                batched()
            torch.cuda.synchronize()
            t_seq, t_bat = [], []
            for _ in range(args.rounds):
                t_seq.append(timed(sequential))
                t_bat.append(timed(batched))
            # the two arms compute the same maps
            a, b = sequential(), batched()
            for s in range(S):
                for name, x, y in zip(("depth", "normal", "mask", "min_sdf"), a[s], b):
                    assert torch.equal(x.detach(), y[s].detach()), (kind, S, s, name)
            ms, mb = statistics.median(t_seq), statistics.median(t_bat)
            print("%-18s %3d  %7.2f [%6.2f, %6.2f]   %7.2f [%6.2f, %6.2f]   %8.2fx  %6.2f -> %6.2f" %
                  (kind, S, ms, min(t_seq), max(t_seq), mb, min(t_bat), max(t_bat), ms / mb,
                   HW * HW / ms / 1e3, HW * HW / mb / 1e3), flush=True)
    print("# maps of the two arms: torch.equal at every (kind, S)")


if __name__ == "__main__":
    main()
