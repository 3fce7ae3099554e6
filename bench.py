#!/usr/bin/env python
"""bench.py -- stylized frames/s at 1280x720 (BASELINE.json metric), one JSON line on stdout.

  python bench.py --gpus N --steps K --warmup W          # this implementation (libfav_b200.so, sm_100a)
  python bench.py --impl reference --gpus N ...           # the reference's CPU nn path (oracle port) on host cores
  python bench.py ... --dump-outputs DIR                  # also write the last timed step's stylized frame to DIR

A "step" = ONE FRAME of the hot path: fused warp+mask+preprocess+concat -> 7-channel input -> stylization net ->
deprocess (run_next_image, fast_artistic_video_core.lua:161-180), recurrent (frame i consumes stylized i-1).
Workload = BASELINE.json configs[1]: 1280x720 clip, candy model (seeded random-init weights of the reference
architecture: no network => no released checkpoints), synthetic frames / flows / certainty masks.

  value      frames/s, inputs resident in HBM, timed with CUDA events on the launching stream, max over ranks
  e2e        frames/s through the host-buffer session API (fav_session_*): every step copies the frame, the
             backward+forward flow from PINNED host memory, computes the occlusion mask on the GPU, and reads
             the stylized frame back to pinned host memory -- all inside the timed region
  roofline   dominant kernel = conv_tc_kernel (tcgen05 implicit GEMM): algorithmic FLOPs / CUDA-event time
  roofline_front  the fused temporal-input kernel (warp-kernel HBM GB/s of the metric), 64 B/px
  cpu_baseline    the oracle port (PyTorch-CPU fp32 restatement + C front end) on the box's host cores
N > 1: one process per GPU (torchrun), independent clips (replicas, weak scaling); NCCL only broadcasts the input
pool from rank 0 before and gathers a checksum after the timed region -- no collective on the data path.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "fast-artistic-videos_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

H, W = 720, 1280
ARCHS = {"default": "c9s1-32,d64,d128,R128,R128,R128,R128,R128,u64,u32,c9s1-3",
         "paper": "c9s1-32,d64,d128,R128,R128,R128,R128,R128,U2,c3s1-64,U2,c9s1-3"}
POOL = 8  # distinct input frames cycled: 8 x 29.5 MB of inputs per rank > 126 MB L2
CONV_GFLOP_720P = 274.3  # SURVEY.md 8(d): logical-channel conv FLOPs per 720p frame, default arch (variant u)
FRONT_BYTES_PER_PX = 64  # fused temporal-input kernel, all-fp32 I/O (SURVEY.md 8(d))
NCU_RES_CONV_DRAM_BYTES = 34215000 + 1113000  # mean of the 10 residual conv_res_kernel launches of one frame, ncu --set full (profiles/r02_frame_raw.csv.gz)
NCU_FRONT_DRAM_BYTES = 33185280 + 586240      # temporal_input_kernel @720p (profiles/r02_frame_raw.csv.gz)
NCU_STAGE_DRAM_BYTES = 37158400 + 1045760      # temporal_stage_kernel<1,0> @720p (profiles/r02_frame_raw.csv.gz)


WORKLOAD = "1280x720 clip (BASELINE.json configs[1]), candy (seeded random-init weights), one step = one frame of run_next_image"


def config_for(arch_key):
    """Identical in both arms (the driver compares the two `config` dicts)."""
    return {"workload": WORKLOAD, "arch": ARCHS[arch_key], "frame": [H, W], "model": "candy (synthetic weights)"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.2 and len(r) >= 9] or [r for (_, r) in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[5 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": reasons, "samples": len(rows),
                "power_w_max": max(float(r[3]) for r in rows)}


def make_pool(n):
    """Synthetic clip segment (SURVEY.md 8(d)): frames, backward/forward flow (u,v)."""
    from fav_b200 import synth

    frames = np.stack([synth.make_frame(H, W, i + 1) for i in range(n)])
    bw = np.stack([synth.make_backward_flow(H, W, i + 2) for i in range(n)])
    fw = np.stack([synth.make_forward_flow(H, W, i + 2) for i in range(n)])
    return frames, bw, fw


# ------------------------------------------------------------------------------------------------------------
def cpu_reference(steps, warmup, budget_s=150.0, arch=None):
    """The reference's CPU nn path, restated (oracle port): C front end + PyTorch-CPU fp32 net, all host threads.
    Each step = one frame of the 720p workload, or a bounded row-strip sample of it when a full frame is too slow
    for the time budget (throughput scaled by the strip fraction; stated in `sample`)."""
    from fav_b200 import synth
    from oracle import net_oracle, pyoracle

    arch = arch or synth.DEFAULT_ARCH
    cores = os.cpu_count() or 1
    ora = net_oracle.NetOracle(style="candy", arch=arch, dtype=torch.float32)

    def one(h, idx, prev):
        frame = synth.make_frame(h, W, 1 + idx % 4)
        flow = synth.checker_to_lua(synth.make_backward_flow(h, W, 2 + idx % 4))
        cert = np.ones((h, W), np.float32)
        cert[h // 3: h // 3 + 32, W // 2: W // 2 + 64] = 0
        t = time.perf_counter()
        cm = pyoracle.min_filter(cert, 7)
        out = ora.run_next_image(frame, prev, flow, cm)
        return time.perf_counter() - t, out.astype(np.float32)

    # give the reference its best thread count (oneDNN / OpenMP often lose with every hardware thread on big hosts)
    cands = sorted({c for c in (cores, cores // 2, 64, 32, 16, 8) if 1 <= c <= cores}, reverse=True)
    best = (None, 1e30)
    for c in cands:
        torch.set_num_threads(c)
        one(96, 0, synth.make_frame(96, W, 1))
        t, _ = one(96, 0, synth.make_frame(96, W, 1))
        if t < best[1]:
            best = (c, t)
    threads = best[0]
    torch.set_num_threads(threads)
    h = H
    t_probe, prev = one(h, 0, synth.make_frame(h, W, 1))
    total = steps + warmup
    if t_probe * total > budget_s:  # bounded sample: a strip of rows (multiple of 4, >= 64)
        h = max(64, int(H * budget_s / (t_probe * total)) // 4 * 4)
        prev = synth.make_frame(h, W, 1)
    for i in range(warmup):
        _, prev = one(h, i, prev)
    t0 = time.perf_counter()
    tt = 0.0
    for i in range(steps):
        dt, prev = one(h, i, prev)
        tt += dt
    wall = time.perf_counter() - t0
    fps = (h / H) * steps / tt
    sample = (f"{steps} frame(s) of rows 0..{h} of the {W}x{H} frame (min_filter + warp/mask/concat + net, fp32), "
              f"{threads} threads (best of {cands} on this {cores}-thread host)" +
              ("" if h == H else "; throughput scaled by the strip fraction"))
    return dict(value=fps, ms_per_step=1e3 * tt / steps * (H / h), cores=threads, sample=sample, wall=wall)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference(args.steps, args.warmup, arch=ARCHS[args.arch])
    line = {"metric": "stylized frames/sec at 1280x720", "impl": "reference", "value": r["value"], "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_for(args.arch),
            "cpu_baseline": {"value": r["value"], "unit": "frames/s", "cores": r["cores"], "kind": "port",
                             "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist

    from fav_b200 import _lib, models_video, session, synth, utils, consistencyChecker

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = utils.bind_host_to_gpu_numa(local)  # before any pinned allocation: host buffers in the GPU's NUMA node
    if world > 1:
        # NCCL prints its version banner on STDOUT at communicator creation; the contract is ONE JSON line on stdout,
        # so fd 1 points at stderr until the final print.
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    K, Wm = args.steps, args.warmup
    pk = peaks()

    arch = ARCHS[args.arch]
    net = models_video.synthetic_model("candy", arch)
    # ---- inputs: rank 0 generates the pool, NCCL broadcast scatters it (the only collective; outside the timed region)
    if rank == 0:
        frames_np, bw_np, fw_np = make_pool(POOL)
        frames, bw, fw = (torch.from_numpy(a).to(dev) for a in (frames_np, bw_np, fw_np))
    else:
        frames = torch.empty((POOL, 3, H, W), device=dev)
        bw = torch.empty((POOL, 2, H, W), device=dev)
        fw = torch.empty((POOL, 2, H, W), device=dev)
    if world > 1:
        for t in (frames, bw, fw):
            dist.broadcast(t, 0)
        frames = torch.roll(frames, rank, 0)  # each rank = an independent clip (different phase of the pool)
        bw, fw = torch.roll(bw, rank, 0), torch.roll(fw, rank, 0)
    flows = torch.stack([bw[:, 1], bw[:, 0]], 1).contiguous()  # (dy,dx) layout of flowFileLoader.lua:31-32
    certs = []
    for i in range(POOL):  # occlusion mask from the flow pair + 7x7 min filter (core.lua:207), on the GPU
        _, c = consistencyChecker.check(bw[i], fw[i], want_cert=True)
        certs.append(utils.min_filter(c, 7))
    certs = torch.stack(certs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # Timed regions: each figure is ONE region of exactly K steps bracketed by barrier + synchronize, so that --steps is the
    # number of timed steps and the last step's inputs (the recurrent state included) are the same from run to run.
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    tw0 = time.time()

    # ---- (1) device-resident throughput: certainty precomputed, frame = fused temporal input + net ---------------------
    prev = net.run_image(frames[0])
    for i in range(Wm):
        j = (i + 1) % POOL
        prev = net.run_next_image(frames[j], prev, flows[j], certs[j])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def region_dev(full):
        nonlocal prev
        barrier()
        l0 = _lib.lib.fav_launch_count()
        e0.record()
        for i in range(K):
            j = (i + 1 + Wm) % POOL
            if full:  # the whole north-star path: occlusion test from the flow pair + 7x7 min filter + warp + net
                _, c = consistencyChecker.check(bw[j], fw[j], want_cert=True)
                c = utils.min_filter(c, 7)
            else:
                c = certs[j]
            prev = net.run_next_image(frames[j], prev, flows[j], c)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1) / 1e3), int(_lib.lib.fav_launch_count() - l0)

    t_dev, launches = region_dev(False)
    out_last = prev  # the stylized frame of the last timed step: what --dump-outputs writes
    checksum = float(prev.double().sum().item())
    value = world * K / t_dev
    t_full = region_dev(True)[0]
    value_full = world * K / t_full

    # ---- (2) end to end through the host-buffer API ------------------------------------------------------------
    sess = session.Session(net, H, W)
    hf = [frames[i].cpu().pin_memory() for i in range(POOL)]
    hbw = [bw[i].cpu().pin_memory() for i in range(POOL)]
    hfw = [fw[i].cpu().pin_memory() for i in range(POOL)]
    hout = [torch.empty((3, H, W)).pin_memory() for _ in range(2)]
    sess.run_image(hf[0], hout[0])
    for i in range(Wm):
        j = (i + 1) % POOL
        sess.run_next_image_flows(hf[j], hbw[j], hfw[j], hout[i & 1], 7)
    sess.sync()

    def region_e2e():
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            j = (i + 1 + Wm) % POOL
            sess.run_next_image_flows(hf[j], hbw[j], hfw[j], hout[i & 1], 7)
        t_enq = time.perf_counter() - t0  # host time to enqueue K frames (copies + launches are asynchronous)
        sess.sync()
        barrier()
        return max_over_ranks(time.perf_counter() - t0), t_enq

    t_e2e, t_enqueue = region_e2e()
    tw1 = time.time()
    clocks = sampler.stop(tw0, tw1) if rank == 0 else None
    gpu_ms_last = sess.last_gpu_ms()
    e2e = world * K / t_e2e
    h2d = (3 + 2 + 2) * H * W * 4
    d2h = 3 * H * W * 4

    # ---- (3) per-kernel breakdown (CUDA events around every plan step) -> roofline -----------------------------
    x7 = torch.empty((1, 7, H, W), device=dev)
    _lib.check(_lib.lib.fav_temporal_input(_lib.dptr(frames[1]), _lib.dptr(prev), _lib.dptr(flows[1]),
                                           _lib.dptr(certs[1]), None, None, _lib.dptr(x7), H, W, 0, _lib.stream_ptr()))
    prof = None
    for _ in range(3):
        prof = net.profile(x7)
    conv_ms = sum(p["ms"] for p in prof if p["kind"] == "conv")
    conv_flop = sum(p["work"] for p in prof if p["kind"] == "conv")
    n_conv_launch = sum(1 for p in prof if p["kind"] == "conv")  # one launch per conv layer (transposed convs: phase-fold)
    stats_ms = sum(p["ms"] for p in prof if p["kind"] == "in_stats")
    apply_ms = sum(p["ms"] for p in prof if p["kind"] == "in_apply")
    pack_ms = sum(p["ms"] for p in prof if p["kind"] == "pack")
    # ---- (4) front-end kernels alone, inputs cycling through the pool (> L2).  A Python loop cannot enqueue 15-us kernels
    # back to back (ctypes call ~10 us), so nf launches are captured into ONE CUDA graph and the replay is timed with events.
    nf = 40
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def graph_ms(launch, reps=5):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(POOL):
                launch(i)
            side.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for i in range(nf):
                    launch(i)
            best = 1e30
            for _ in range(reps):
                f0.record(side)
                g.replay()
                f1.record(side)
                side.synchronize()
                best = min(best, f0.elapsed_time(f1) / nf)
        torch.cuda.current_stream().wait_stream(side)
        return best

    out7 = torch.empty((7, H, W), device=dev)
    # (a) fused warp + mask + preprocess + concat with a given certainty plane (64 B/px, SURVEY 8d)
    front_ms = graph_ms(lambda i: _lib.check(_lib.lib.fav_temporal_input(
        _lib.dptr(frames[i % POOL]), _lib.dptr(frames[(i + 3) % POOL]), _lib.dptr(flows[i % POOL]), _lib.dptr(certs[i % POOL]), None, None,
        _lib.dptr(out7), H, W, 0, _lib.stream_ptr())))
    front_gbs = FRONT_BYTES_PER_PX * H * W / (front_ms * 1e-3) / 1e9
    # (b) the WHOLE temporal stage in one kernel: occlusion test from the flow pair + 7x7 min filter + (a): 68 B/px (SURVEY 8d)
    stage_ms = graph_ms(lambda i: _lib.check(_lib.lib.fav_temporal_stage(
        _lib.dptr(frames[i % POOL]), _lib.dptr(frames[(i + 3) % POOL]), _lib.dptr(flows[i % POOL]), _lib.dptr(fw[i % POOL]), None, None, None,
        _lib.dptr(out7), None, H, W, 7, 0, _lib.stream_ptr())))
    stage_gbs = 68 * H * W / (stage_ms * 1e-3) / 1e9
    # (c) standalone warp op (metric half 2: warp-kernel HBM GB/s, 32 B/px) and the kernel to beat: the reference's own CUDA
    # kernel compiled for sm_100a (oracle/_ref/libref_warp.so, original 32x16 blocks), same inputs, real and stress flows
    warp = {}
    if rank == 0:
        from oracle import refwarp

        stress = torch.from_numpy(np.stack([synth.stress_flow(H, W, seed=7 + i) for i in range(POOL)])).to(dev)
        wout = torch.empty((1, 3, H, W), device=dev)
        imgs4, flows4, stress4 = frames[:, None], flows[:, None], stress[:, None]
        have_ref = refwarp.available()
        wbytes = 32 * H * W
        for kind, fl in (("real", flows4), ("stress", stress4)):
            ms_o = graph_ms(lambda i: _lib.check(_lib.lib.fav_warp_image(_lib.dptr(imgs4[i % POOL]), 3, H, W, _lib.dptr(fl[(i + 3) % POOL]),
                                                                         H, W, _lib.dptr(wout), 0, _lib.stream_ptr())))
            ms_r = graph_ms(lambda i: refwarp.warp(imgs4[i % POOL], fl[(i + 3) % POOL], wout)) if have_ref else None
            warp[kind] = {"ms": ms_o, "gbs": wbytes / (ms_o * 1e-3) / 1e9,
                          "original_kernel_ms": ms_r, "original_kernel_gbs": (wbytes / (ms_r * 1e-3) / 1e9) if ms_r else None,
                          "vs_original_kernel": (ms_r / ms_o) if ms_r else None}
    conv_tfs = conv_flop / (conv_ms * 1e-3) / 1e12
    res = [p for p in prof if p["kind"] == "conv" and (".c1" in p["name"] or ".c2" in p["name"])]
    res_ms, res_flop, res_n = sum(p["ms"] for p in res), sum(p["work"] for p in res), len(res)
    res_tfs = res_flop / (res_ms * 1e-3) / 1e12 if res else conv_tfs

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_reference(2, 1, budget_s=25.0, arch=arch)
        cpu = {"value": r["value"], "unit": "frames/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}

    if world > 1:
        cs = torch.tensor([checksum], dtype=torch.float64, device=dev)
        gathered = [torch.zeros_like(cs) for _ in range(world)]
        dist.all_gather(gathered, cs)  # "gather outputs": one checksum per clip
    if rank == 0:
        line = {
            "metric": "stylized frames/sec at 1280x720", "value": value, "value_full": value_full, "unit": "frames/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": 1e3 * t_dev / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16x2 (fp16 hi/lo operand pairs, 3 tcgen05 MMAs per product, fp32 accumulate)",
            "data": "synthetic",
            "config": config_for(args.arch),
            "notes": {"l2": f"inputs cycle through a pool of {POOL} distinct frames ({POOL * 29.5:.0f} MB > 126 MB L2); "
                            "~1.5 GB of activations stream through L2 per frame",
                      "parallelism": f"replicas x{world} (independent clips, no data-path collective)",
                      "precision": "outputs within 1e-3 of the fp64 oracle (measured ~1e-5, tests/test_gpu_net.py, "
                                   "tests/test_gpu_parity_large.py)",
                      "timing": f"one timed region of exactly {K} steps per figure (barrier + synchronize on both sides, max "
                                "over ranks); value / value_full: CUDA events, e2e: host clock"},
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * t_e2e / K, "host_enqueue_ms_per_step": 1e3 * t_enqueue / K,
                    "gpu_ms_last_frame": gpu_ms_last,
                    "note": "fav_session_run_next_image_flows: frame + bw/fw flow from pinned host memory, occlusion "
                            "mask + min filter + warp + net on the GPU, stylized frame back to pinned host memory"},
            "gpu_launches": launches,
            "clocks": clocks,
            "host": {"gpu_numa_binding": numa},
            "roofline": {"bound": "tensor",
                         "kernel": "conv_res_kernel, residual-block launches (128->128 3x3; 10 of the %d conv launches per " % n_conv_launch +
                                   "frame, the largest share of the step; the second conv of each block also normalises its input on load)",
                         "achieved": res_tfs, "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": res_tfs / pk["tf_sust"],
                         "traffic": NCU_RES_CONV_DRAM_BYTES,
                         "traffic_source": "profiles/r02_frame_raw.csv.gz (dram__bytes_read.sum + dram__bytes_write.sum, mean of the 10 "
                                           "launches of one frame; algorithmic bytes per launch 68.5 MB: the planar raw output stays in L2)",
                         "peak_source": pk["src"] + ", bf16 sustained (kernel timed inside the step)",
                         "algorithmic_flop_per_launch": res_flop / max(1, res_n), "us_per_launch": 1e3 * res_ms / max(1, res_n),
                         "launches_timed": res_n,
                         "all_conv_launches": {"achieved": conv_tfs, "frac": conv_tfs / pk["tf_sust"],
                                               "algorithmic_flop_per_frame": conv_flop, "launches_per_frame": n_conv_launch,
                                               "ms_per_frame": conv_ms},
                         "note": "algorithmic (logical fp32) FLOPs; the fp16 hi/lo scheme executes 3x that on the tensor "
                                 "pipe (3 MMAs per product), so executed-MMA utilisation is 3x frac and frac <= 1/3"},
            "roofline_stage": {"bound": "hbm", "kernel": "temporal_stage_kernel<false,0> (the whole temporal stage in one launch: "
                               "occlusion test from the flow pair + 7x7 min filter + warp + mask + preprocess + concat)",
                               "achieved": stage_gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": stage_gbs / pk["hbm"],
                               "bytes_per_launch": 68 * H * W, "ms": stage_ms, "traffic": NCU_STAGE_DRAM_BYTES,
                               "traffic_source": "profiles/r02_frame_raw.csv.gz (37.2 MB read = the input planes; the packed operand it "
                                                 "writes stays in L2); not memory bound: the occlusion test's mixed float/double chain",
                               "timing": f"{nf} launches in one CUDA graph, inputs cycle through {POOL} frames, best of 5 replays"},
            "roofline_front": {"bound": "hbm", "kernel": "temporal_input_kernel (fused warp+mask+preprocess+concat)",
                               "achieved": front_gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": front_gbs / pk["hbm"],
                               "traffic": NCU_FRONT_DRAM_BYTES,
                               "traffic_source": "profiles/r02_frame_raw.csv.gz (33.2 MB read = exactly the input planes; "
                                                 "the 25.8 MB written stay in the 126 MB L2)",
                               "bytes_per_launch": FRONT_BYTES_PER_PX * H * W, "ms": front_ms},
            "roofline_warp": None if not warp else {
                "bound": "hbm", "kernel": "warp_vec4_kernel<3> via fav_warp_image (nn.BilinearSamplerBDHW forward, 3x720x1280)",
                "achieved": warp["real"]["gbs"], "peak": pk["hbm"], "unit": "GB/s", "frac": warp["real"]["gbs"] / pk["hbm"],
                "bytes_per_launch": 32 * H * W, "traffic": None,
                "vs_original_kernel": warp["real"]["vs_original_kernel"],
                "real_flow": warp["real"], "stress_flow_u64px": warp["stress"],
                "original_kernel": "stnbdhw/BilinearSamplerBDHW.cu:48-109 compiled for sm_100a from /root/reference "
                                   "(oracle/Makefile refwarp), launch config of :119-120"},
            "value_full_note": "value_full = device-resident frames/s with the occlusion test (flow pair) and the 7x7 min filter "
                               "inside the timed region as well (the whole north-star path; `value` takes precomputed certainty)",
            "breakdown_ms_per_frame": {"conv": conv_ms, "in_stats": stats_ms, "in_apply": apply_ms, "pack_input": pack_ms,
                                       "temporal_input": front_ms, "total_device": 1e3 * t_dev / K,
                                       "total_device_full_path": 1e3 * t_full / K},
            "layers": [{"name": p["name"], "kind": p["kind"], "ms": round(p["ms"], 4),
                        **({"tflops": round(p["work"] / (p["ms"] * 1e-3) / 1e12, 1)} if p["kind"] == "conv" else
                           {"gbs": round(p["work"] / (p["ms"] * 1e-3) / 1e9, 1)})} for p in prof],
            "cpu_baseline": cpu,
            "checksum": checksum,
        }
        if world > 1:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        if world > 1:
            os.dup2(2, 1)
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "stylized_frame.npy"), out_last.cpu().numpy())
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------
def run_cfg3(args):
    """BASELINE.json configs[2]: 8 independent 1920x1080 clips data-parallel over N GPUs.  Rank 0 owns every clip's decoded
    inputs in PINNED HOST memory (frames + backward/forward flow, fp32); fav_b200.clips.stream_clips uploads them chunk by
    chunk, sends them to the owning ranks over NCCL (batch_isend_irecv), each rank runs its clips' recurrent loops
    (fav_run_next_image_flows: occlusion test + min filter + warp + net per frame) and sends the stylized chunks back; rank 0
    copies them to pinned host memory.  EVERYTHING is inside the timed region."""
    import torch.distributed as dist

    from fav_b200 import clips, models_video, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from fav_b200 import utils as fav_utils

    numa = fav_utils.bind_host_to_gpu_numa(local)  # before any pinned allocation: host buffers in the GPU's NUMA node
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)  # NCCL banner must not reach stdout
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    else:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1"); os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("gloo", rank=0, world_size=1)  # N = 1: the data plane degenerates to local uploads
    Hc, Wc, NC, CH, PO = 1080, 1920, 8, 4, 4
    F = max(8, args.steps)
    net = models_video.synthetic_model("candy", ARCHS[args.arch])
    state = {}
    host = {}
    bytes_mode = args.payload == "bytes"
    fr = np.stack([synth.make_frame(Hc, Wc, i + 1) for i in range(PO)])
    fw = np.stack([synth.make_forward_flow(Hc, Wc, i + 2) for i in range(PO)])
    if bytes_mode:
        # what the files hold: 8-bit frames (P6 payload, HWC) and the backward .flo payload ((u,v) pairs); converted on the owner GPU
        fr = np.ascontiguousarray(np.clip(np.rint(fr * 255.0), 0, 255).astype(np.uint8).transpose(0, 2, 3, 1))
        bw = np.stack([np.ascontiguousarray(synth.make_backward_flow(Hc, Wc, i + 2).transpose(1, 2, 0)) for i in range(PO)])
        out_shape, out_dtype = (Hc, 1 + 3 * Wc), torch.uint8  # image.save's 8-bit pixels as Sub-filtered PNG scanlines
    else:
        bw = np.stack([synth.checker_to_lua(synth.make_backward_flow(Hc, Wc, i + 2)) for i in range(PO)])  # (dy,dx), flowFileLoader.lua:31-32
        out_shape, out_dtype = (3, Hc, Wc), torch.float32
    pool = (("fr", fr), ("bw", bw), ("fw", fw))
    in_shapes = [tuple(v.shape[1:]) for _, v in pool]
    in_dtypes = [torch.from_numpy(v[:1]).dtype for _, v in pool]
    dpool = {k: torch.from_numpy(v).to(dev) for k, v in pool}  # compute-only leg (every rank)
    if rank == 0:
        host = {k: torch.from_numpy(v).pin_memory() for k, v in pool}
        out_host = [torch.empty((CH,) + out_shape, dtype=out_dtype).pin_memory() for _ in range(NC)]

    def load_chunk(c, f0, f1):
        # H2D straight from the pinned decoded pool into a device chunk (no host-side staging copy)
        idx = [(c + i) % PO for i in range(f0, f1)]
        res = []
        for k in ("fr", "bw", "fw"):
            buf = torch.empty((len(idx),) + tuple(host[k].shape[1:]), dtype=host[k].dtype, device=dev)
            for i, j in enumerate(idx):
                buf[i].copy_(host[k][j], non_blocking=True)
            res.append(buf)
        return res

    def process_chunk(c, f0, inputs):
        fr_, bw_, fw_ = inputs
        outs = []
        for i in range(fr_.shape[0]):
            if bytes_mode:
                content, flow, _ = fav_utils.bytes_to_planes(fr_[i], bw_[i])
            else:
                content, flow = fr_[i], bw_[i]
            if f0 + i == 0:
                prev = net.run_image(content)
            else:
                prev = net.run_next_image_flows(content, state[c], flow, fw_[i], None, 7)
            state[c] = prev
            outs.append(fav_utils.planes_to_png_rows(prev) if bytes_mode else prev)
        return torch.stack(outs)

    def store_chunk(c, f0, out):
        out_host[c][: out.shape[0]].copy_(out, non_blocking=True)

    def timed(fn):
        """barrier + synchronize on both sides; the time is taken ON THE DEVICE (events on the compute stream, which joins the
        transfer streams before the closing event); max over ranks is taken by the caller"""
        state.clear()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st = fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return e0.elapsed_time(e1) * 1e-3, st

    def run(nf):
        return timed(lambda: clips.stream_clips(NC, nf, CH, in_shapes, out_shape, load_chunk, process_chunk, store_chunk, device=dev,
                                                in_dtypes=in_dtypes, out_dtype=out_dtype))

    def run_compute_only(nf):
        """the same clips and frame loops with every input already resident on the owning GPU: what the data plane costs
        is the difference to run()"""
        mine = [c for c in range(NC) if clips.owner(c, world) == rank]

        def body():
            for k in range(0, nf, CH):
                for c in mine:
                    idx = [(c + i) % PO for i in range(k, min(nf, k + CH))]
                    process_chunk(c, k, [dpool[key][idx] for key in ("fr", "bw", "fw")])
            return None
        return timed(body)

    h2d_gbps = None
    if rank == 0:  # what this box's PCIe link delivers from pinned memory (256 MB, outside the timed region)
        probe_h, probe_d = torch.empty(64 << 20, dtype=torch.float32).pin_memory(), torch.empty(64 << 20, dtype=torch.float32, device=dev)
        probe_d.copy_(probe_h, non_blocking=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); probe_d.copy_(probe_h, non_blocking=True); e1.record(); torch.cuda.synchronize()
        h2d_gbps = probe_h.numel() * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9
        del probe_h, probe_d
    run(2 * CH)  # warm-up: plans, graphs, NCCL connections
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    tw0 = time.time()
    t, st = run(F)
    tw1 = time.time()
    run_compute_only(2 * CH)
    tc, _ = run_compute_only(F)
    tt = torch.tensor([t, tc], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_max, tc_max = float(tt[0]), float(tt[1])
    if rank == 0:
        clocks = sampler.stop(tw0, tw1)
        per_frame_in = sum(int(np.prod(v.shape[1:])) * v.itemsize for _, v in pool)
        per_frame_out = int(np.prod(out_shape)) * (1 if bytes_mode else 4)
        line = {"metric": "stylized frames/sec, 8 independent 1920x1080 clips (BASELINE.json configs[2])", "value": NC * F / t_max,
                "unit": "frames/s", "n_gpus": world, "steps": F, "warmup": 2 * CH, "ms_per_step": 1e3 * t_max / F,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f16x2 (fp16 hi/lo operand pairs, 3 tcgen05 MMAs per product, fp32 accumulate)", "data": "synthetic",
                "config": {"workload": "8 x 1920x1080 clips, candy (synthetic weights), one step = one frame of EVERY clip",
                           "arch": ARCHS[args.arch], "frames_per_clip": F, "chunk": CH,
                           "parallelism": f"clips round-robin over {world} GPU(s); rank 0 scatters inputs / gathers outputs (NCCL p2p)"},
                "data_plane": {"payload": args.payload,
                               "source": "rank 0 pinned host memory: " + ("8-bit frames as the files hold them + backward .flo payload + forward "
                                         "flow planes; byte->float / (u,v)->(dy,dx) on the owning GPU (fav_bytes_to_planes); results return as "
                                         "8-bit Sub-filtered PNG scanlines (fav_planes_to_png_rows = image.save's quantisation)" if bytes_mode
                                         else "fp32 frames + bw/fw flow, fp32 stylized frames back"),
                               "bytes_in_per_frame": per_frame_in, "bytes_out_per_frame": per_frame_out, "nccl_bytes_sent_rank0": st["bytes_in"],
                               "compute_only_frames_per_s": NC * F / tc_max, "compute_only_ms_per_step": 1e3 * tc_max / F,
                               "data_plane_exposed_share": max(0.0, 1.0 - tc_max / t_max),
                               "streams": "uploads + NCCL on a transfer stream, D2H of results on a third, frame loops on the compute stream",
                               "rank0_h2d_GBps_needed": NC * F * per_frame_in / t_max / 1e9, "rank0_h2d_GBps_probe": h2d_gbps,
                               "gpu_numa_binding": numa,
                               "limit": "every input byte crosses rank 0's single PCIe link (H2D) before NVLink: the scatter is "
                                        "bound by that link, not by NVLink / NVSwitch"},
                "clocks": clocks}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3"],
                    help="cfg2 = BASELINE.json configs[1] (the metric: 1280x720 clip, default); cfg3 = configs[2]: 8 x 1080p clips "
                         "with the NCCL scatter / gather of frames inside the timed region")
    ap.add_argument("--payload", default="bytes", choices=["bytes", "fp32"],
                    help="cfg3 only: what travels from rank 0 to the owning GPU and back: the 8-bit pixels the files hold (converted on "
                         "the GPU; default) or decoded fp32 tensors")
    ap.add_argument("--arch", default="default", choices=list(ARCHS),
                    help="default = train_video.lua:21 (u64,u32); paper = README.md:256 (U2,c3s1-64,U2)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the stylized frame of the last timed step (rank 0) as "
                         "DIR/stylized_frame.npy (float32, 3xHxW); the inputs are the same from run to run")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config != "cfg2"):
        ap.error("--dump-outputs applies to the default workload (--impl ours --config cfg2)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "cfg3":
        run_cfg3(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
