#!/usr/bin/env python
"""bench.py -- net_forward images/sec @256x256 (BASELINE.json metric) + p50 single-click latency.

    python bench.py --gpus N --steps K --warmup W            # this framework (one rank per GPU)
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU path

A step = ONE forward of the hot path (pack+conv1_1 -> conv trunk -> regression head) over one batch of synthetic
256x256 L + sparse-hint inputs (BASELINE config 3: 64 images / GPU, weak scaling).
  value    images/s with the inputs resident in HBM: K replays of the CUDA-graph-captured forward (the shipped
           configuration: no per-op events, kernels chained by programmatic dependent launch), device-timed with CUDA
           events, max over ranks.  Per-op times come from a SEPARATE, untimed profiling pass.
  e2e      the same through the host-pointer C-ABI call (pinned H2D of the inputs + D2H of the ab maps inside the
           timed region).
  config4  BASELINE config 4 as an extra record at every --gpus N: 512x512, GLOBAL batch 16 with a global-hints
           vector per image, sharded 16/N per GPU (strong scaling: 1 vs 8 GPUs).
  latency  BASELINE config 5 (20 sequential put_point -> forward, dist head on): p50/p99 of the complete click at the
           C ABI (announced click: forward + the clicked pixel's pmf + 9 colour suggestions from ONE graph launch), the
           round-2 protocol next to it (unannounced_*), and the wrapper-level calls the GUI makes (ui/gui_draw.py:258-286)
           with two separate models and with the launcher's shared trunk.
Every rank also runs ONE fixed-seed image outside the timed region; rank 0 asserts that all ranks produced the same
bytes (the rank != 0 weight path: reserve -> broadcast -> adopt).
--dump-outputs DIR writes rank 0's ab maps of the last timed step to DIR/ab.npy (float32 [N,2,X,X]; only the leading
images when the batch exceeds 60 MiB).  Weights and inputs are seeded, so two builds run with the same arguments can be
compared output for output.
The reference arm times the UNMODIFIED reference wrapper `ColorizeImageTorch.net_forward` (staged by
`__graft_entry__.build()` into the git-ignored oracle/_ref/, kind "reference") on the host cores, looping single-image
calls as the reference does (models/pytorch/model.py:139-141); without the staged copy it falls back to the CPU oracle
port (oracle/lhn_ref.py, kind "port").
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "net_forward images/sec @256x256"   # --size 512 reports the same metric name with the size in config
X = 256
PER_GPU_BATCH = 64
DUMP_BYTES = 60 << 20                        # --dump-outputs stays under 64 MB, .npy header included
NCU_TRAFFIC_CSV = os.path.join(ROOT, "profiles", "r02_ncu_full_batch64_forward.csv")


def _ncu_traffic(batch, size):
    """dram__bytes_read + dram__bytes_write per launch of the dominant kernel (mean over the 25 umma_conv launches of
    the regression trunk), from the committed `ncu --set full` capture of this same workload at HEAD
    (profiles/r02_ncu_full_batch64_forward.csv, written by tools/ncu_summary.py)."""
    if batch != 64 or size != 256 or not os.path.isfile(NCU_TRAFFIC_CSV):
        return None
    import csv
    rows = list(csv.reader(l for l in open(NCU_TRAFFIC_CSV) if not l.startswith("#")))
    h = rows[0]
    tot, n = 0.0, 0
    for r in rows[1:]:
        d = dict(zip(h, r))
        if d["kernel"].startswith("umma_conv_kernel") and d["op"] != "class":
            tot += (float(d["dram_read_MB"]) + float(d["dram_write_MB"])) * 1e6
            n += 1
    return tot / n if n else None


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"tensor": d.get("bf16_tflops_sustained", 1370.8), "tensor_burst": d.get("bf16_tflops", 1653.3),
                "hbm": d.get("hbm_gbs", 6569.6), "src": "measured (MEASURED_PEAKS.json, sustained bf16 cuBLAS)"}
    return {"tensor": 1400.0, "tensor_burst": 1590.0, "hbm": 6650.0, "src": "fallback (B200_PROFILING.md)"}


def workload_config(N, size, world):
    """`config` of the JSON line -- identical for both arms (the reference arm describes its bounded sample in
    cpu_baseline.sample, not here)."""
    return {"workload": "BASELINE config %s: %d x %dx%d synthetic L + 0-10 sparse 7x7 ab hints per GPU, "
                        "regression head (ab map)" % ("3" if size == 256 else "4 (no global hints)", N, size, size),
            "per_gpu_batch": N, "global_batch": N * world,
            "parallelism": "dp%d (image sharding, no per-step collective)" % world,
            "l2_policy": "per-step working set (~%.1f GB of activations) >> 126 MB L2; inputs are not re-used from L2"
                         % (N * 0.15 * (size / 256.0) ** 2)}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index=0):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.samples, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                f = [s.strip() for s in line.split(",")]
                if len(f) >= 6 and f[0].isdigit():
                    self.samples.append((time.perf_counter(), f))
        except Exception:
            pass

    def finish(self, t_begin=None, t_end=None):
        """Only samples taken inside [t_begin, t_end] (the timed region) count."""
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        allf = [f for _, f in self.samples]
        inside = [f for t, f in self.samples if (t_begin is None or t >= t_begin) and (t_end is None or t <= t_end)]
        self.samples = inside if inside else allf
        sm = [int(s[0]) for s in self.samples]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": int(statistics.median(sm)) if sm else None,
                "sm_max_mhz": int(self.samples[0][1]) if self.samples else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "power_w_median": (statistics.median([float(s[6]) for s in self.samples if len(s) > 6 and s[6].replace(".", "").isdigit()])
                                   if any(len(s) > 6 for s in self.samples) else None)}


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference's own code when staged (oracle/_ref), else the oracle port
# ----------------------------------------------------------------------------------------------
class CpuArm(object):
    """One single-image CPU forward per call, as the reference runs it (batch 1, models/pytorch/model.py:139-141)."""

    def __init__(self):
        import torch
        from oracle import ref_shims, synth
        self.torch, self.synth = torch, synth
        self.sd = synth.torch_state_dict(1234)
        self.kind = "port"
        self.cm = None
        if ref_shims.reference_available():
            try:
                import tempfile
                CI = ref_shims.import_reference_wrapper()
                wpath = os.path.join(tempfile.mkdtemp(), "synthetic_1234.pth")
                torch.save(self.sd, wpath)
                import contextlib
                import io
                with contextlib.redirect_stdout(io.StringIO()):
                    cm = CI.ColorizeImageTorch(Xd=X, maskcent=True)
                    cm.prep_net(path=wpath)
                    cm.set_image(np.random.RandomState(0).randint(0, 256, (X, X, 3)).astype(np.uint8))
                self.cm, self.kind = cm, "reference"
            except Exception as e:                      # staged copy unusable: fall back to the port, say why
                sys.stderr.write("reference wrapper unavailable (%r): timing the oracle port\n" % (e,))
        self.L, self.ab, self.m = synth.synthetic_batch(8, X, seed=0, max_hints=10)

    def describe(self):
        if self.kind == "reference":
            return ("the UNMODIFIED reference ColorizeImageTorch.net_forward (data/colorize_image.py:249-268: net forward with "
                    "autograd on as the reference calls it + Lab->RGB + RGB->Lab post-process), staged in oracle/_ref")
        return "CPU oracle port of SIGGRAPHGenerator.forward (oracle/lhn_ref.py, torch fp32, no_grad, no post-process)"

    def one(self, i):
        i %= self.L.shape[0]
        if self.cm is not None:
            self.cm.net_forward(self.ab[i].astype(np.float64), self.m[i].astype(np.float64))
        else:
            from oracle import lhn_ref
            with self.torch.no_grad():
                lhn_ref.lhn_forward(self.sd, self.L[i:i + 1], self.ab[i:i + 1], self.m[i:i + 1], 0.5)

    def run(self, budget_s, max_images, nthreads=None):
        """-> (images/s, images, threads)"""
        if nthreads:
            self.torch.set_num_threads(nthreads)
        self.one(0)                                      # warm-up (oneDNN primitive cache)
        t0, n = time.perf_counter(), 0
        while n < max_images and (time.perf_counter() - t0) < budget_s:
            self.one(n)
            n += 1
        return n / (time.perf_counter() - t0), n, self.torch.get_num_threads()

    def best_threads(self):
        """The reference uses torch's default thread pool; on a 128-core host the default (all cores) is pathologically
        slow for batch-1 convs, so the baseline runs at the best of a few pool sizes (favours the reference)."""
        ncpu = os.cpu_count() or 1
        best = (0.0, ncpu)
        for t in sorted(set([min(ncpu, c) for c in (8, 16, 32, 64)] + [ncpu])):
            ips, _, _ = self.run(4.0, 2, t)
            if ips > best[0]:
                best = (ips, t)
        return best[1]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    global X
    X = args.size
    arm = CpuArm()
    nthr = arm.best_threads()
    per_step = 4                       # bounded sample: 4 single-image CPU forwards per step
    for _ in range(args.warmup):
        arm.run(1e9, 1, nthr)
    t0 = time.perf_counter()
    n = 0
    for _ in range(args.steps):
        _, k, thr = arm.run(1e9, per_step, nthr)
        n += k
    dt = time.perf_counter() - t0
    ips = n / dt
    line = {"impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.batch, X, args.gpus),
            "cpu_baseline": {"value": ips, "unit": "images/s", "cores": thr, "kind": arm.kind,
                             "sample": "bounded: %d single-image calls per step (%d images in all) of %s; images drawn from the "
                                       "config-3 workload (the reference has no batch API); best-of pool sizes -> %d threads of %d "
                                       "host cores" % (per_step, n, arm.describe(), thr, os.cpu_count() or 0)},
            "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def timed_graph_steps(torch, ctx, fwd, steps, warmup, barrier, dev):
    """Capture ONE forward into a CUDA graph (torch capture of the stream the C ABI launches on) and time `steps`
    replays with CUDA events.  Falls back to plain stream launches if capture is refused.  -> (ms_total, mode)"""
    mode = "cuda graph replay (torch.cuda.graph capture of idc_forward; kernels chained by PDL)"
    graph = None
    try:
        s = torch.cuda.Stream(dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            fwd()
        torch.cuda.current_stream(dev).wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            fwd()
    except Exception as e:
        sys.stderr.write("graph capture refused (%r): timing stream launches\n" % (e,))
        graph, mode = None, "stream launches (kernels chained by PDL)"
        torch.cuda.synchronize(dev)
    run = graph.replay if graph is not None else fwd
    for _ in range(max(warmup, 3)):
        run()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        run()
    e1.record()
    barrier()
    t1 = time.perf_counter()
    return e0.elapsed_time(e1), mode, (t0, t1)


def run_config4(args, torch, dist, world, rank, local, dev, barrier, max_over_ranks):
    """BASELINE config 4: 512x512, global batch 16, global-hints vector per image, 16/world images per GPU."""
    from interactive_deep_colorization_b200.parallel import ShardedColorizer, shard_range
    from oracle import caffe_spec, synth
    G, S = 16, 512
    start, count = shard_range(G, world, rank)
    sd = None
    if rank == 0 or world == 1:
        sd = synth.torch_state_dict(1234)
        sd.update({k: torch.from_numpy(v) for k, v in caffe_spec.synthetic_glob_state_dict().items()})
    eng = ShardedColorizer(S, S, max(count, 1), state_dict=sd, device=local, dist_head=False, use_graph=False,
                           global_hints=True)
    ctx = eng.ctx
    L, ab, m = synth.synthetic_batch(G, S, seed=40, max_hints=10)          # the same 16 images on every rank ...
    ga, sat = synth.synthetic_glob(G, seed=3)
    glob = np.ascontiguousarray(np.concatenate([ga, sat], axis=1).astype(np.float32))
    sl = slice(start, start + count)                                         # ... each rank takes its slice
    hL, hab, hm, hg = (torch.from_numpy(np.ascontiguousarray(a[sl])).pin_memory() for a in (L, ab, m, glob))
    dL, dab, dm, dg = hL.to(dev), hab.to(dev), hm.to(dev), hg.to(dev)
    out = torch.empty((count, 2, S, S), dtype=torch.float32, device=dev)
    hout = torch.empty((count, 2, S, S), dtype=torch.float32).pin_memory()
    ms_total, mode, _ = timed_graph_steps(torch, ctx, lambda: ctx.forward_device(dL, dab, dm, 0.5, glob=dg, out_ab=out),
                                          args.steps, args.warmup, barrier, dev)
    ms_step = max_over_ranks(ms_total, dev) / args.steps
    for _ in range(2):
        ctx.forward_host(hL.numpy(), hab.numpy(), hm.numpy(), 0.5, glob=hg.numpy(), out_ab=hout.numpy())
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ctx.forward_host(hL.numpy(), hab.numpy(), hm.numpy(), 0.5, glob=hg.numpy(), out_ab=hout.numpy())
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0, dev)
    flops = ctx.flops_per_image()
    ctx.close()
    return {"workload": "BASELINE config 4: 512x512, GLOBAL batch 16 with a 316-entry global-hints vector per image, "
                        "sharded %d image(s) per GPU over %d GPU(s)" % (count, world),
            "value": G / (ms_step * 1e-3), "unit": "images/s", "ms_per_step": ms_step, "scaling": "strong",
            "global_batch": G, "per_gpu_batch": count, "n_gpus": world,
            "e2e": {"value": G * args.steps / e2e_s, "unit": "images/s",
                    "h2d_bytes_per_step": int(G * (4 * S * S + 316) * 4), "d2h_bytes_per_step": int(G * 2 * S * S * 4)},
            "useful_tflops": G * flops / (ms_step * 1e-3) / 1e12, "launch_mode": mode}


def run_latency(local, L):
    """BASELINE config 5 at two levels: the C-ABI click call and the wrapper calls the GUI makes."""
    from interactive_deep_colorization_b200 import colorize_image as CI
    from interactive_deep_colorization_b200.engine import LhnContext
    from oracle import synth
    sd = synth.torch_state_dict(1234)
    lctx = LhnContext(device=local, max_n=1, H=X, W=X, dist=True)
    lctx.load_state_dict(sd)
    lctx.set_dist_resident(True)      # config 5: the click only needs dist[:, h//4, w//4]
    rs = np.random.RandomState(0)
    l1 = np.ascontiguousarray(L[:1]); a1 = np.zeros((1, 2, X, X), np.float32); m1 = np.zeros((1, 1, X, X), np.float32)
    times, reccs_times = [], []
    for i in range(25):
        loc = rs.randint(8, X - 8, 2)
        CI.put_point(a1[0], m1[0], loc, 3, rs.uniform(-80, 80, 2))
        t = time.perf_counter()
        lctx.forward_host(l1, a1, m1, 0.5, want_rgb=True)
        lctx.fetch_dist(0, int(loc[0]) // 4, int(loc[1]) // 4)
        times.append((time.perf_counter() - t) * 1e3)
        t = time.perf_counter()       # not part of config 5: the K=9 colour suggestions the GUI shows (row f2)
        lctx.ab_reccs(0, int(loc[0]) // 4, int(loc[1]) // 4, K=9)
        reccs_times.append((time.perf_counter() - t) * 1e3)
    pageable = times[5:]
    # the same clicks with the context's page-locked click buffers (LhnContext.click_buffers / idc_host_alloc): the
    # copy nodes of the graph read / write the caller's memory, no CPU staging copy
    buf = lctx.click_buffers(1)
    buf["L_mc"][...] = l1
    buf["ab"][...] = 0
    buf["mask"][...] = 0
    times = []
    for i in range(25):
        loc = rs.randint(8, X - 8, 2)
        CI.put_point(buf["ab"][0], buf["mask"][0], loc, 3, rs.uniform(-80, 80, 2))
        t = time.perf_counter()
        lctx.forward_host(buf["L_mc"], buf["ab"], buf["mask"], 0.5, want_rgb=True, out_ab=buf["out_ab"], out_rgb=buf["out_rgb"])
        lctx.fetch_dist(0, int(loc[0]) // 4, int(loc[1]) // 4)
        times.append((time.perf_counter() - t) * 1e3)
    unannounced = times[5:]
    # the shipped click: the image is resident (idc_set_image, once per photo -- the reference's set_image / net_forward
    # split), the click is announced (idc_set_click) so its pmf AND the K=9 suggestions ride on the dist head's side
    # branch of the same graph; everything the GUI shows after a click is inside the timed region
    lctx.set_image(buf["L_mc"])
    times = []
    for i in range(25):
        loc = rs.randint(8, X - 8, 2)
        CI.put_point(buf["ab"][0], buf["mask"][0], loc, 3, rs.uniform(-80, 80, 2))
        y4, x4 = int(loc[0]) // 4, int(loc[1]) // 4
        t = time.perf_counter()
        lctx.set_click(0, y4, x4, 9)
        lctx.forward_host(None, buf["ab"], buf["mask"], 0.5, want_rgb=True, out_ab=buf["out_ab"], out_rgb=buf["out_rgb"])
        lctx.fetch_dist(0, y4, x4)
        lctx.ab_reccs(0, y4, x4, K=9)
        times.append((time.perf_counter() - t) * 1e3)
    times = times[5:]
    lat = {"p50_ms": float(np.percentile(times, 50)), "p99_ms": float(np.percentile(times, 99)),
           "unannounced_p50_ms": float(np.percentile(unannounced, 50)), "unannounced_p99_ms": float(np.percentile(unannounced, 99)),
           "pageable_p50_ms": float(np.percentile(pageable, 50)), "pageable_p99_ms": float(np.percentile(pageable, 99)),
           "reccs_k9_p50_ms": float(np.percentile(reccs_times[5:], 50)), "calls": len(times),
           "what": "BASELINE config 5: put_point -> idc_set_click (pixel + K=9) -> C-ABI idc_forward_host (batch 1, resident "
                   "image, dist head + Lab->RGB on, one CUDA graph: H2D of the hints, PDL-chained kernels, the dist head + the "
                   "clicked pixel's pmf + its 9 colour suggestions on a side branch, D2H of ab + rgb) -> idc_fetch_dist + "
                   "idc_ab_reccs (host-side reads); page-locked click buffers.  unannounced_*: round-2 protocol (L re-sent, "
                   "pmf fetched by a separate device call, no suggestions; reccs_k9 = what a separate suggestion call costs). "
                   "pageable_*: ordinary numpy arrays (staged by the CPU)"}
    lctx.close()
    # wrapper level, as ui/gui_draw.py:258-286 calls it: colour model net_forward (RGB + quantised output_ab),
    # dist model net_forward + get_ab_reccs (predict_color / suggest_color)
    import contextlib
    import io
    img = np.random.RandomState(1).randint(0, 256, (X, X, 3)).astype(np.uint8)

    def pair(shared):
        with contextlib.redirect_stdout(io.StringIO()):
            cm = CI.ColorizeImageB200(Xd=X, maskcent=True)
            cm.prep_net(state_dict=sd, dist=shared)
            cd = CI.ColorizeImageB200Dist(Xd=X, maskcent=True)
            if shared:
                cd.share_trunk(cm)        # launcher --backend b200: one checkpoint, one trunk (ideepcolor.py:34-38)
            else:
                cd.prep_net(state_dict=sd)
        cm.set_image(img); cd.set_image(img)
        ab64, m64 = np.zeros((2, X, X)), np.zeros((1, X, X))
        t_col, t_all = [], []
        for i in range(25):
            loc = rs.randint(8, X - 8, 2)
            CI.put_point(ab64, m64, loc, 3, rs.uniform(-80, 80, 2))
            t = time.perf_counter()
            if shared:
                cd.hint_click(int(loc[0]), int(loc[1]), K=9)
            cm.net_forward(ab64, m64)
            t1 = time.perf_counter()
            cd.net_forward(ab64, m64)
            cd.get_ab_reccs(int(loc[0]), int(loc[1]), K=9)
            t2 = time.perf_counter()
            t_col.append((t1 - t) * 1e3); t_all.append((t2 - t) * 1e3)
        return t_col[5:], t_all[5:]
    t_col, t_all = pair(False)
    lat["wrapper_p50_ms"] = float(np.percentile(t_col, 50))
    lat["wrapper_p99_ms"] = float(np.percentile(t_col, 99))
    lat["wrapper_with_dist_reccs_p50_ms"] = float(np.percentile(t_all, 50))
    _, t_pair = pair(True)
    lat["wrapper_shared_trunk_with_dist_reccs_p50_ms"] = float(np.percentile(t_pair, 50))
    lat["wrapper_what"] = ("ColorizeImageB200.net_forward(ab, mask) -> uint8 RGB + quantised output_ab (float64 numpy in/out, one "
                           "C-ABI call); with_dist_reccs adds ColorizeImageB200Dist.net_forward + get_ab_reccs(K=9) on a second "
                           "context, as ui/gui_draw.py:258-286 calls them; shared_trunk = the launcher's default pairing "
                           "(ColorizeImageB200Dist.share_trunk + hint_click): the same three calls, ONE forward")
    return lat


def run_ours(args):
    import torch
    import torch.distributed as dist
    from interactive_deep_colorization_b200.parallel import ShardedColorizer, max_over_ranks
    from oracle import synth            # cpu_baseline leg + synthetic weights/inputs only

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    N = args.batch
    global X
    X = args.size
    sd = synth.torch_state_dict(1234) if rank == 0 or world == 1 else None
    eng = ShardedColorizer(X, X, N, state_dict=sd, device=local, dist_head=False, use_graph=False,
                           fast_fp16=args.fast_fp16)
    ctx = eng.ctx
    # per-rank synthetic inputs (config 3), distinct seeds per rank
    L, ab, m = synth.synthetic_batch(N, X, seed=1000 * rank, max_hints=10)
    hL = torch.from_numpy(L).pin_memory(); hab = torch.from_numpy(ab).pin_memory(); hm = torch.from_numpy(m).pin_memory()
    dL, dab, dm = hL.to(dev), hab.to(dev), hm.to(dev)
    out = torch.empty((N, 2, X, X), dtype=torch.float32, device=dev)
    hout = torch.empty((N, 2, X, X), dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- every rank: one fixed-seed image, checksum compared on rank 0 (rank != 0 weight path) ----
    cL, cab, cm_ = synth.synthetic_batch(1, X, seed=424242, max_hints=10)
    cout = ctx.forward_device(torch.from_numpy(cL).to(dev), torch.from_numpy(cab).to(dev), torch.from_numpy(cm_).to(dev), 0.5)["ab"]
    torch.cuda.synchronize(dev)
    hc = cout.cpu().numpy()                                 # checksums on the host: no library kernel on the GPU
    csum = torch.tensor([float(hc.astype(np.float64).sum()), float(np.abs(hc.astype(np.float64)).sum()),
                         float((hc.view(np.int32).astype(np.int64) & 0xFFFF).sum())], dtype=torch.float64, device=dev)
    if world > 1:
        allsums = [torch.zeros_like(csum) for _ in range(world)]
        dist.all_gather(allsums, csum)
    else:
        allsums = [csum]
    ranks_equal = all(bool(torch.equal(allsums[0], s)) for s in allsums)
    if rank == 0 and not ranks_equal:
        raise RuntimeError("rank outputs differ on the fixed-seed image: %r" % ([s.tolist() for s in allsums],))

    # ---- device-resident throughput: graph replays, no profiling inside the timed region ----
    ctx.forward_device(dL, dab, dm, 0.5, out_ab=out)
    launches_per_step = ctx.last_launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    ms_total, launch_mode, (t_region0, t_region1) = timed_graph_steps(
        torch, ctx, lambda: ctx.forward_device(dL, dab, dm, 0.5, out_ab=out), args.steps, args.warmup, barrier, dev)
    ms_total = max_over_ranks(ms_total, dev)
    clocks = sampler.finish(t_region0, t_region1) if sampler else None
    ms_step = ms_total / args.steps
    value = world * N / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:
        ab_last = out.cpu().numpy()
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "ab.npy"), ab_last[:DUMP_BYTES // ab_last[0].nbytes])

    # ---- per-op device times: separate untimed pass (events between the launches, PDL off by construction) ----
    ctx.set_profiling(True)
    for _ in range(3):
        ctx.forward_device(dL, dab, dm, 0.5, out_ab=out)
    prof = ctx.get_profile()
    ctx.set_profiling(False)

    # ---- end to end through the host-pointer C-ABI call (pinned H2D + forward + D2H) ----
    e2e = None
    if not args.skip_e2e:
        for _ in range(2):
            ctx.forward_host(hL.numpy(), hab.numpy(), hm.numpy(), 0.5, out_ab=hout.numpy())
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ctx.forward_host(hL.numpy(), hab.numpy(), hm.numpy(), 0.5, out_ab=hout.numpy())
        barrier()
        e2e_s = max_over_ranks(time.perf_counter() - t0, dev)
        e2e = world * N * args.steps / e2e_s
    flops_img = ctx.flops_per_image()
    ctx.close()
    del dL, dab, dm, out
    torch.cuda.empty_cache()

    # ---- BASELINE config 4 (512^2, global batch 16, global hints) at this N ----
    cfg4 = None
    if not args.skip_e2e and not args.no_config4 and X == 256 and not args.fast_fp16:
        cfg4 = run_config4(args, torch, dist, world, rank, local, dev, barrier, max_over_ranks)

    # ---- single-click latency (config 5): 20 sequential put_point -> net_forward, batch 1 ----
    lat = None
    if rank == 0 and not args.skip_e2e:
        lat = run_latency(local, L)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel (umma_conv_kernel: every conv/deconv layer of the trunk) ----
    peaks = _peaks()
    conv = [(n, ms, f) for (n, ms, f) in prof[1:-1]]
    conv_ms = sum(ms for _, ms, _ in conv)
    conv_flops = sum(f for _, _, f in conv) * N
    achieved = conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
    n_launch = sum(1 for _ in conv)
    split = 1.0 if args.fast_fp16 else 3.0
    roofline = {"bound": "tensor", "kernel": "umma_conv_kernel<BN,MT,CG,SPLIT,HALO> (tcgen05 implicit-GEMM conv, %d launches/step)" % n_launch,
                "achieved": achieved, "peak": peaks["tensor"], "unit": "TFLOP/s", "frac": achieved / peaks["tensor"],
                "issued_mma_frac": split * achieved / peaks["tensor"],
                "peak_source": peaks["src"], "traffic": _ncu_traffic(N, X),
                "traffic_note": "average DRAM bytes per umma_conv launch (ncu --set full at HEAD, profiles/%s)" % os.path.basename(NCU_TRAFFIC_CSV),
                "algorithmic_flops_per_launch": conv_flops / max(n_launch, 1),
                "avg_launch_ms": conv_ms / max(n_launch, 1),
                "kernel_share_of_step": min(1.0, conv_ms / ms_step),
                "whole_step_useful_tflops_per_gpu": N * flops_img / (ms_step * 1e-3) / 1e12,
                "note": "achieved = useful conv FLOPs (2*MACs) / summed per-launch device time from the untimed profiling pass; "
                        "the split-FP16 scheme issues 3 MMAs per product, so the tensor pipe is busy issued_mma_frac of peak"}
    # ---- CPU baseline (bounded sample, rank 0, N=1 only) ----
    cpu = None
    if world == 1 and not args.no_cpu_baseline and not args.skip_e2e:
        arm = CpuArm()
        ips, nimg, thr = arm.run(15.0, 64, arm.best_threads())
        cpu = {"value": ips, "unit": "images/s", "cores": thr, "kind": arm.kind,
               "sample": "%d images @%dx%d, batch-1 loop of %s (best-of pool sizes -> %d threads, %d host cores)"
                         % (nimg, X, X, arm.describe(), thr, os.cpu_count() or 0)}
        if lat:
            lat["cpu_ms_per_image"] = 1e3 / ips
            lat["speedup_vs_cpu_latency"] = (1e3 / ips) / lat["p50_ms"]
    line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": ("f16 operands single pass (NOT parity: ~6e-2 ab error), f32 accumulate" if args.fast_fp16 else
                      "f16x2-split operands, f32 accumulate (ab within 1e-3 of the f32 reference)"),
            "data": "synthetic",
            "config": workload_config(N, X, world),
            "launch_mode": launch_mode,
            "roofline": roofline, "cpu_baseline": cpu,
            "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": int(world * N * 4 * X * X * 4),
                    "d2h_bytes_per_step": int(world * N * 2 * X * X * 4)},      # whole job, all ranks
            "gpu_launches": world * launches_per_step * args.steps, "clocks": clocks, "latency": lat,
            "config4": cfg4, "rank_outputs_identical": ranks_equal,
            "per_op_ms": {n: round(ms, 4) for n, ms, _ in prof}}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="images per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config4", action="store_true", help="skip the extra BASELINE config 4 record")
    ap.add_argument("--size", type=int, default=256, help="image side")
    ap.add_argument("--fast-fp16", action="store_true",
                    help="NOT the parity configuration: single-pass FP16 operands (1 MMA per product, ~6e-2 ab error)")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only: skip the e2e, config 4 and latency legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's ab maps to DIR/ab.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: use it with --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
