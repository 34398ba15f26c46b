#!/usr/bin/env python
"""bench.py -- rays/s of the sphere-tracing hot path (BASELINE.json metric) on N GPUs of one node.

  python bench.py --gpus N --steps K --warmup W          (N>1: launched under torch.distributed.run)
  python bench.py --impl reference ...                   (CPU arm: the oracle port of the reference, rank 0 only)
  python bench.py ... --dump-outputs DIR                 (also writes the last timed step's outputs to DIR/*.npy)

A "step" is one full differentiable render of the metric's workload -- SDFRenderer.render() of ONE 512x512 image (depth +
normal + silhouette, 50-step 'recursive' march, buffer 5) with gradients enabled w.r.t. the 256-d latent, a scalar loss
and backward() -- on synthetic inputs (seeded geometric-init 8x512 DeepSDF decoder, seeded latent, fixed camera).
At N GPUs the SAME 512x512 image is split N ways (interleaved bands of 4-row groups, 262144/N rays per GPU: STRONG
scaling, the configuration BASELINE.json's metric names at 1/2/4/8 GPUs); the bands and the partial latent gradients are
exchanged with ONE all-gather per step (21 B/ray).  Extra keys, not the headline:
  `weak`     the round-1 weak-scaling number (image side round(512 sqrt N), ~262144 rays per GPU);
  `config5`  BASELINE config 5: 2048x2048 forward depth+normal render, tile-sharded over the N GPUs + the all-gather;
  `per_rank` min / max over ranks of: step, decoder kernels, pack, all-gather (incl. waiting for the slowest rank), unpack.

`value`   : rays/s with inputs resident in HBM (CUDA events, max over ranks).
`e2e`     : same metric through the public API with HOST buffers: H2D of latent/R/T from pinned memory and D2H of
            all four output maps + the latent gradient inside the timed region.
`roofline`: the decoder-row kernel (dominant) event-timed inside the running step; achieved = useful flops
            (F = 3,146,752 per folded decoder row, 2F per gradient row) / kernel time, against the measured dense bf16
            peak of MEASURED_PEAKS.json.
"""
import argparse
import gc
import importlib
import json
import math
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

HW_BASE = 512
MARCH_STEP, BUFFER = 50, 5
KIND = "recursive"
CPU_SAMPLE_HW = 192


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


def loss_of(out):
    """A scalar of the rendered maps: depth summed over the silhouette + the min-|sdf| map (gradients reach every sample
    the renderer selected).  Written with torch.where rather than boolean indexing: indexing would size its result on the
    host, i.e. stall the stream in the middle of every step."""
    depth, normal, mask, min_sdf = out
    return torch.where(mask.bool(), depth, torch.zeros_like(depth)).sum() + min_sdf.sum()


class ClockSampler(object):
    """NVML sampling (background thread, 20 ms period) of SM clocks, power and throttle reasons during the timed
    region.  NVML in-process instead of an `nvidia-smi -lms` subprocess: the subprocess costs ~100 ms per sample and
    measurably slows a 50-80 ms step."""

    def __init__(self, index):
        self.index, self.rows, self.stop, self.th, self.h, self.nv = index, [], False, None, None, None

    def __enter__(self):
        try:
            if self.index < 0:
                raise RuntimeError('sampler disabled')
            import threading
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)

            def run():
                while not self.stop:
                    try:
                        self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                          nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0,
                                          nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
                    except Exception:
                        pass
                    time.sleep(0.02)
            self.th = threading.Thread(target=run, daemon=True)
            self.th.start()
        except Exception:
            self.th = None
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.th is not None:
            self.th.join(timeout=2)

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.rows:
            return out
        nv = self.nv
        out["sm_mhz"] = statistics.median(r[0] for r in self.rows)
        out["sm_max_mhz"] = self.max_sm
        out["power_w_max"] = max(r[1] for r in self.rows)
        out["samples"] = len(self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[2]
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        out["reasons"] = [k for k, v in names.items() if bits & v]
        return out


def weak_side(n_gpus):
    return int(round(HW_BASE * math.sqrt(n_gpus)))


def cpu_render_step(ren, lat, R, T):
    l = lat.clone().requires_grad_(True)
    out = ren.render(l, R, T, ray_marching_type=KIND)
    loss_of(out).backward()
    return l.grad


def run_reference(args, rank, world):
    """CPU arm.  The reference is pure Python/PyTorch and its tree is absent on the GPU box, so what is timed is the
    oracle port (oracle/sdf_oracle.py: the same PyTorch ops in the same order, pinned bit for bit to the reference where
    the reference exists) on the host cores -- `cpu_baseline.kind = "port"`.  Workload = this bench's own (`config`): a
    512x512 fwd+bwd render per step costs 40-60 s of CPU, so each step renders a BOUNDED SAMPLE of it: the same view at
    SxS pixels, S the largest of 512/384/256/192/128 whose K+W steps fit ~4 minutes (estimated from one 128x128 probe;
    CPU rays/s does not depend on the image size: the decoder GEMMs dominate).  The sample is stated in `sample`,
    `config.cpu_sample` and `cpu_baseline.sample`; warm-up and step counts are the ones asked for."""
    if rank != 0:
        return
    from oracle.sdf_oracle import OracleSDFRenderer
    synth = importlib.import_module("dist-renderer_b200.synth")
    cores = pick_threads(synth)
    dec = synth.make_decoder("B")
    R, T = synth.front_camera()
    lat = synth.make_latent()

    def renderer(S):
        return OracleSDFRenderer(dec, synth.intrinsic(S, S), img_hw=(S, S), march_step=MARCH_STEP, buffer_size=BUFFER)
    t0 = time.time()
    cpu_render_step(renderer(128), lat, R, T)
    probe = time.time() - t0
    budget = float(os.environ.get("BENCH_CPU_BUDGET_S", "240")) / max(1, args.steps + args.warmup)
    S = 128
    for cand in (512, 384, 256, 192):
        if probe * (cand / 128.0) ** 2 * 1.1 <= budget:
            S = cand
            break
    ren = renderer(S)
    for _ in range(args.warmup):
        cpu_render_step(ren, lat, R, T)
    t0 = time.time()
    for _ in range(args.steps):
        cpu_render_step(ren, lat, R, T)
    dt = time.time() - t0
    value = S * S * args.steps / dt
    sample = ("each step renders the workload's view at %dx%d (%s of its 512x512 rays) fwd+bwd with the oracle port, %d torch "
              "threads of %d host cores" % (S, S, "all" if S == 512 else "1/%d" % ((512 * 512) // (S * S)), cores, os.cpu_count() or 1))
    cfg = config_of(args.gpus)
    cfg["cpu_sample"] = "%dx%d" % (S, S)
    line = {
        "impl": "reference", "metric": "rays/sec (fwd+bwd)", "value": value, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg, "sample": sample,
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


def pick_threads(synth):
    """Thread count that gives the oracle's decoder GEMMs the best throughput on this host (many-core boxes lose badly
    to oversubscription at os.cpu_count() threads).  Best of three timings per candidate so the choice is stable."""
    dec = synth.make_decoder("B")
    x = torch.cat([synth.make_latent().expand(20000, -1), torch.rand(20000, 3) - 0.5], 1)
    cores = os.cpu_count() or 1
    best = (None, 1)
    for n in sorted(set(min(cores, c) for c in (8, 16, 32, 64))):
        torch.set_num_threads(n)
        with torch.no_grad():
            dec.inference(x[:2000])
            dt = None
            for _ in range(3):
                t0 = time.time()
                dec.inference(x)
                d = time.time() - t0
                dt = d if dt is None else min(dt, d)
        if best[0] is None or dt < 0.95 * best[0]:      # a larger count has to win clearly
            best = (dt, n)
    torch.set_num_threads(best[1])
    return best[1]


def cpu_port_baseline(synth, lat_h, R_h, T_h):
    """Oracle port of the reference on the host cores, bounded sample (~10-30 s): the workload's view at 192x192, fwd+bwd."""
    from oracle.sdf_oracle import OracleSDFRenderer
    threads = pick_threads(synth)
    dec_c = synth.make_decoder("B")
    Hc = CPU_SAMPLE_HW
    ora = OracleSDFRenderer(dec_c, synth.intrinsic(Hc, Hc), img_hw=(Hc, Hc), march_step=MARCH_STEP, buffer_size=BUFFER)
    t0 = time.time()
    cpu_render_step(ora, lat_h, R_h, T_h)
    dt = time.time() - t0
    return {"value": Hc * Hc / dt, "unit": "rays/s", "cores": threads, "kind": "port",
            "sample": "the workload's view at %dx%d (1/%d of its rays) fwd+bwd, once, %d torch threads of %d host cores "
                      "(best of a thread sweep)" % (Hc, Hc, 512 * 512 // (Hc * Hc), threads, os.cpu_count() or 1)}


def dump_outputs(path, result):
    """The result of the last timed step as its caller receives it -- the four full-image maps of render() and the
    gradient w.r.t. the latent -- one float32 .npy per array (6.3 MB at 512x512), for comparing builds output by output.
    The maps repeat bit for bit from run to run; the latent gradient is summed with float atomics and moved by ~4e-7
    rel-L2 between runs on one B200."""
    import numpy as np
    (depth, normal, mask, min_sdf), latent_grad = result
    os.makedirs(path, exist_ok=True)
    for name, t in (("depth", depth), ("normal", normal), ("mask", mask), ("min_sdf", min_sdf), ("latent_grad", latent_grad)):
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def config_of(n_gpus, side=HW_BASE):
    return {"workload": "%dx%d render(): depth+normal+silhouette, single shape (geometric-init 8x512 DeepSDF, 256-d "
                        "latent), %d-step '%s' march, buffer %d, fwd + backward over the latent"
                        % (side, side, MARCH_STEP, KIND, BUFFER),
            "rays_per_gpu": side * side // n_gpus,
            "parallelism": "ray-tile: the image split %d ways (interleaved bands of 4-row groups), one all-gather" % n_gpus,
            "l2": "flushed between timed iterations (256 MiB write)"}


def ncu_traffic(tc):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, from the committed `ncu --set full`
    capture (profiles/r2_tc_raw.csv, row 3: mlp_tc_kernel<0> on a dense march step's mix of 262,144 rows, 60 % in the
    one-pass segment); None when no capture is committed (the fp32 engine has none this round)."""
    import csv
    if not tc:
        return None
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r2_tc_raw.csv")
    try:
        rows = list(csv.reader(open(path)))
        unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        col = {h: i for i, h in enumerate(rows[0])}
        r = rows[4]
        assert "mlp_tc_kernel<0>" in r[col["Kernel Name"]]
        return sum(float(r[col[k]]) * unit[rows[1][col[k]]] for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
    except Exception:
        return None


_JSON_OUT = None


def _emit(line):
    """The one JSON line of the contract, on the process's ORIGINAL stdout."""
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # stdout carries exactly one JSON line: NCCL prints its version banner (and INFO lines) with printf on fd 1 whatever
    # NCCL_DEBUG_FILE says, so fd 1 is pointed at stderr for the whole run and the JSON goes to a saved copy of the real stdout
    global _JSON_OUT
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--engine", default="auto")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the weak-scaling and config-5 extra measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    assert world == args.gpus or world == 1, "launch with torch.distributed.run --nproc-per-node N for --gpus N"
    import ctypes
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pkg = importlib.import_module("dist-renderer_b200")
    synth = importlib.import_module("dist-renderer_b200.synth")
    par = importlib.import_module("dist-renderer_b200.parallel")
    abi = importlib.import_module("dist-renderer_b200._abi")
    __import__("__graft_entry__").build()
    lib = abi.lib()

    side = HW_BASE
    dec = synth.make_decoder("B").to(dev)
    R_h, T_h = synth.front_camera()
    lat_h = synth.make_latent()
    flush = torch.empty(64 * 1024 * 1024, device=dev, dtype=torch.float32)  # 256 MiB > 126 MB L2
    lat_d, R_d, T_d = lat_h.to(dev), R_h.to(dev), T_h.to(dev)
    n_lat = lat_h.numel()

    def sharded(s):
        return par.ShardedSDFRenderer(dec, synth.intrinsic(s, s), (s, s), rank=rank, world_size=world, march_step=MARCH_STEP,
                                      buffer_size=BUFFER, engine=args.engine)
    ren = sharded(side)

    def make_step(r, grad=True, check=False):
        def step(lat_src, R_src, T_src):
            if not grad:
                out = r.render(lat_src, R_src, T_src, ray_marching_type=KIND, no_grad=True)
                return r.gather(out, check_empty=check)[0], None
            lat = lat_src.detach().requires_grad_(True)
            out = r.render(lat, R_src, T_src, ray_marching_type=KIND)
            loss_of(out).backward()
            full, extras = r.gather(out, extra=lat.grad, check_empty=check)
            return full, extras.sum(0)
        return step
    step_device = make_step(ren)

    def timed(fn, steps, warmup):
        """Device time of `steps` calls (max over ranks), barrier + synchronize on both sides, L2 flushed between calls."""
        for _ in range(warmup):
            fn()
            flush.fill_(1.0)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        marks = []
        for _ in range(steps):
            fn()
            flush.fill_(1.0)
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            marks.append(ev)
        b.record()
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        per = [round((a if i == 0 else marks[i - 1]).elapsed_time(marks[i]), 2) for i in range(len(marks))]
        return float(t.item()), per

    # ---- device-resident timing (the headline `value`)
    for _ in range(args.warmup):
        step_device(lat_d, R_d, T_d)
        flush.fill_(1.0)
    torch.cuda.synchronize()
    ren.local.reset_row_counter()
    gc.collect()
    gc.disable()   # no cyclic-GC pauses inside the timed regions (re-enabled below)
    l0 = lib.dist_launch_count()
    last = [None]

    def headline_step():
        last[0] = step_device(lat_d, R_d, T_d)
    with ClockSampler(local_rank if not os.environ.get('BENCH_NO_SAMPLER') else -1) as clk:
        ms, step_ms = timed(headline_step, args.steps, 0)
    launches = lib.dist_launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last[0])
    last[0] = None
    rows_f = int(ren.local.rows_evaluated.item())
    rows_g, rows_gc = [int(v) for v in ren.local.rows_grad.tolist()]     # full gradient rows (2F), mask-cache replays (F)
    tiles_1p, tiles_3p = [int(v) / args.steps for v in ren.local.tile_counters.tolist()]
    value = side * side * args.steps / (ms * 1e-3)
    clocks = clk.summary()

    # ---- the same steps once more with every decoder-kernel launch bracketed by CUDA events on its stream
    # (dist_profile_begin/end) and events around pack / all-gather / unpack: where a rank's step time goes
    n_prof = max(1, min(args.steps, 5))
    ren.local.reset_row_counter()
    ren.events = {}
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    abi.check(lib.dist_profile_begin())
    p0 = torch.cuda.Event(enable_timing=True); p1 = torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(n_prof):
        step_device(lat_d, R_d, T_d)
        flush.fill_(1.0)
    p1.record()
    torch.cuda.synchronize()
    k_total_ms, k_launches = ctypes.c_double(0.0), ctypes.c_longlong(0)
    abi.check(lib.dist_profile_end(ctypes.byref(k_total_ms), ctypes.byref(k_launches)))
    ev = ren.events
    ren.events = None
    span = lambda a, b: sum(x.elapsed_time(y) for x, y in zip(ev[a], ev[b])) / n_prof
    prof = {"steps": n_prof, "step_ms": p0.elapsed_time(p1) / n_prof, "kernel_ms": k_total_ms.value / n_prof,
            "launches": k_launches.value / n_prof, "rows_f": int(ren.local.rows_evaluated.item()) / n_prof,
            "rows_g": int(ren.local.rows_grad[0].item()) / n_prof, "rows_gc": int(ren.local.rows_grad[1].item()) / n_prof,
            "tiles_1p": int(ren.local.tile_counters[0].item()) / n_prof, "tiles_3p": int(ren.local.tile_counters[1].item()) / n_prof,
            "pack_ms": span("pack0", "pack1"), "gather_ms": span("pack1", "gather1"), "unpack_ms": span("gather1", "unpack1")}
    keys = ("step_ms", "kernel_ms", "pack_ms", "gather_ms", "unpack_ms")
    mine = torch.tensor([prof[k] for k in keys], device=dev)
    allr = mine[None]
    if world > 1:
        allr = torch.empty(world, len(keys), device=dev)
        dist.all_gather_into_tensor(allr, mine[None].contiguous())
    per_rank = {k: {"min": round(float(allr[:, i].min()), 3), "max": round(float(allr[:, i].max()), 3)} for i, k in enumerate(keys)}
    per_rank["other_ms"] = {"min": round(float((allr[:, 0] - allr[:, 1:].sum(1)).min()), 3),
                            "max": round(float((allr[:, 0] - allr[:, 1:].sum(1)).max()), 3)}
    per_rank["note"] = ("per step, %d profiled steps after the timed region: decoder kernels (CUDA events around each launch), "
                        "pack, all-gather (includes waiting for the slowest rank), unpack; other = march update / set-up kernels, "
                        "host-side autograd + launch gaps, L2 flush" % n_prof)

    # ---- end to end through the public API with host buffers
    pin = lambda x: x.clone().pin_memory()
    lat_p, R_p, T_p = pin(lat_h), pin(R_h), pin(T_h)
    outs_p = [torch.empty(side, side).pin_memory(), torch.empty(side, side, 3).pin_memory(),
              torch.empty(side, side, dtype=torch.uint8).pin_memory(), torch.empty(side, side).pin_memory()]
    g_p = torch.empty(n_lat).pin_memory()
    step_checked = make_step(ren, check=True)

    def step_e2e():
        full, g = step_checked(lat_p.to(dev, non_blocking=True), R_p.to(dev, non_blocking=True),
                               T_p.to(dev, non_blocking=True))
        if rank == 0:
            for dst, src in zip(outs_p, full):
                dst.copy_(src, non_blocking=True)
            g_p.copy_(g.reshape(-1), non_blocking=True)
        torch.cuda.synchronize()

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        step_e2e()
        flush.fill_(1.0)
    e1.record()
    torch.cuda.synchronize()
    ms_e = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    t = torch.tensor([ms_e], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_e = float(t.item())
    e2e_value = side * side * args.steps / (ms_e * 1e-3)
    h2d = (lat_p.numel() + R_p.numel() + T_p.numel()) * 4
    d2h = sum(o.numel() * o.element_size() for o in outs_p) + g_p.numel() * 4

    # ---- extras: round-1 style weak scaling, and BASELINE config 5 (2048x2048 forward, sharded over the N GPUs)
    extras = {}
    if not args.no_extras:
        n_x = max(2, min(args.steps, 5))
        if world > 1:
            sw = weak_side(world)
            rw = sharded(sw)
            sd = make_step(rw)
            ms_w, _ = timed(lambda: sd(lat_d, R_d, T_d), n_x, 2)
            extras["weak"] = {"value": sw * sw * n_x / (ms_w * 1e-3), "unit": "rays/s", "ms_per_step": ms_w / n_x, "steps": n_x,
                              "workload": "%dx%d fwd+bwd (image side 512 sqrt N: ~262144 rays per GPU), as in round 1" % (sw, sw)}
            del rw, sd
        r5 = sharded(2048)
        s5 = make_step(r5, grad=False)
        ms_5, _ = timed(lambda: s5(lat_d, R_d, T_d), n_x, 1)
        extras["config5"] = {"value": 2048 * 2048 * n_x / (ms_5 * 1e-3), "unit": "rays/s (forward)", "ms_per_step": ms_5 / n_x,
                             "steps": n_x, "workload": "2048x2048 forward depth+normal+silhouette render, %d-step '%s' march, "
                             "tile-sharded over %d GPU(s) + one all-gather of the output bands" % (MARCH_STEP, KIND, world)}
        del r5, s5
    gc.enable()

    # ---- roofline of the dominant kernel: decoder rows, timed alone (rank 0)
    F = ren.local.flops_per_row()
    roof = None
    cpu_baseline = None
    if rank == 0:
        peak_burst, peak_sust, _, src = load_peaks()
        n_rows = 262144
        gen = torch.Generator().manual_seed(11)
        pts = ((torch.rand(n_rows, 3, generator=gen) - 0.5) * 1.2).to(dev)
        for _ in range(2):
            pkg.decode_sdf(dec, lat_d, pts, clamp_dist=None, no_grad=True, engine=args.engine)
        reps = 5
        torch.cuda.synchronize()
        time.sleep(1.5)     # "timed alone": let the power-capped clocks of the long timed loops above recover
        e0.record()
        for _ in range(reps):
            pkg.decode_sdf(dec, lat_d, pts, clamp_dist=None, no_grad=True, engine=args.engine)
        e1.record()
        torch.cuda.synchronize()
        k_ms = e0.elapsed_time(e1) / reps
        isolated = n_rows * F / (k_ms * 1e-3) / 1e12
        in_step = (rows_f * F + rows_g * 2 * F + rows_gc * F) / (ms * 1e-3) / 1e12
        # dominant kernel inside the step: useful flops of its launches / their summed event-timed durations.  A backward row
        # replayed from the mask cache runs the transposed chain only: F, not 2F
        achieved = (prof["rows_f"] * F + prof["rows_g"] * 2 * F + prof["rows_gc"] * F) / (prof["kernel_ms"] * 1e-3) / 1e12
        tc_on = ren.local.plan.tc is not None
        passes = 3 if tc_on else 1
        # MMA flops actually issued by the decoder kernels per step: forward tile programs (128 rows each, padding rows
        # included) with one or three fp16 passes, gradient rows (forward + transposed chain) always with three
        issued = ((prof["tiles_1p"] + 3 * prof["tiles_3p"]) * 128 * F + (2 * prof["rows_g"] + prof["rows_gc"]) * 3 * F) if tc_on else \
            (prof["rows_f"] + 2 * prof["rows_g"]) * F
        issued_tf = issued / (prof["kernel_ms"] * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": achieved, "peak": peak_sust, "unit": "TFLOP/s",
                "frac": achieved / peak_sust, "traffic": ncu_traffic(ren.local.plan.tc is not None),
                "peak_source": src + " dense bf16, sustained (kernel timed inside the running step)",
                "kernel": "decoder-row tile kernel: %.0f launches/step, %.1f us average, %.1f %% of the step (CUDA events "
                          "around every launch, %d extra steps after the timed region)"
                          % (prof["launches"], 1e3 * prof["kernel_ms"] / max(prof["launches"], 1),
                             100.0 * prof["kernel_ms"] / prof["step_ms"], prof["steps"]),
                "flop_per_row": F, "launches_per_step": prof["launches"], "kernel_ms_per_step": prof["kernel_ms"],
                "kernel_share_of_step": prof["kernel_ms"] / prof["step_ms"],
                "issued_tflops": issued_tf, "issued_frac": issued_tf / peak_sust,
                "two_tier": {"tiles_one_pass_per_step": prof["tiles_1p"], "tiles_three_pass_per_step": prof["tiles_3p"],
                             "note": "forward 128-row tile programs of the march (re-queries and coarse pyramid levels "
                                     "included); a screened tile that fails is counted in both"},
                "isolated": {"tflops": isolated, "rows_per_launch": n_rows, "ms_per_launch": k_ms,
                             "frac_of_burst_peak": isolated / peak_burst, "issued_frac_of_burst_peak": passes * isolated / peak_burst,
                             "burst_peak": peak_burst,
                             "note": "one 262,144-row forward launch at full split precision (3 fp16 MMA passes), after a cooldown"},
                "traffic_note": "dram bytes of one 262,144-row launch with a dense march step's tier mix (ncu --set full, profiles/r2_tc_raw.csv)",
                "note": "achieved counts USEFUL flops (F per folded decoder row, 2F per gradient row, F per backward row replayed "
                        "from the forward's ReLU-mask cache, which runs the transposed chain only) over the event-timed "
                        "decoder kernels of the running step; the tensor-core engine issues 3 fp16 MMA passes per logical GEMM "
                        "(split-fp16, fp32-level parity) on rows that need them",
                "whole_step_tflops": in_step, "rows_fwd_per_step": rows_f / args.steps, "rows_grad_per_step": rows_g / args.steps,
                "rows_grad_from_mask_cache_per_step": rows_gc / args.steps}
        # ---- CPU baseline (oracle port) on a bounded sample, rank 0 at N=1 only
        if world == 1 and not args.no_cpu_baseline:
            cpu_baseline = cpu_port_baseline(synth, lat_h, R_h, T_h)
    if rank == 0:
        line = {
            "metric": "rays/sec (fwd+bwd)", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32 (split-fp16 tensor-core operands, fp32 accumulate)"
            if ren.local.plan.tc is not None else "f32", "data": "synthetic",
            "config": config_of(world), "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e / args.steps},
            "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu_baseline,
            "engine": "tc" if ren.local.plan.tc is not None else "simt", "step_ms": step_ms, "per_rank": per_rank,
        }
        line.update(extras)
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
