#!/usr/bin/env python
"""Benchmark of the OpenIBL hot path on B200 (see DESIGN.md).

    python bench.py [--gpus N --steps K --warmup W]          # B200 engine (libiblb200.so)
    python bench.py --impl reference [...]                   # reference CPU arithmetic (oracle port)
    python bench.py [...] --dump-outputs DIR                 # also save what the timed calls returned

Primary metric (BASELINE.json): images/sec of VGG16+NetVLAD+PCA descriptor extraction at batch 32,
3x480x640 synthetic images (configs[1]).  The same JSON line carries the retrieval metric
(query x database pairs/sec, 6.8k x 10k x 4096-d, configs[2]) under "retrieval".
A step = one batch of 32 images through the whole extraction path; --steps K times exactly K of them.

--dump-outputs DIR writes rank 0's results of the last timed step as DIR/<name>.npy (1.3 MB in all):
descriptors.npy (float32 [32, 4096], Engine.extract with PCA) and retrieval_topk_dist.npy /
retrieval_topk_idx.npy (float32 / float64 [6800, 10], sharded_topk).  Inputs and weights are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GFLOP_PER_IMAGE_BACKBONE = 187.92        # SURVEY 8(a1), 480x640
BATCH = 32
H, W = 480, 640
NQ, NDB, DIM, TOPK = 6800, 10000, 4096, 10


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.startswith("Active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def load_conv_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the 12 conv3x3_tc_kernel launches of one batch-32 step, from
    the ncu capture committed under profiles/ (per-layer table with layer labels; tools/ncu_conv_traffic.py made it)."""
    p = os.path.join(ROOT, "profiles", "r02_conv_traffic.json")
    if not os.path.exists(p):
        return {"dram_bytes_per_step": None, "note": "no ncu traffic table committed (profiles/r02_conv_traffic.json)"}
    t = json.load(open(p))
    if os.environ.get("IBL_CONV1_FUSED", "1") != "0" and "dram_bytes_total_with_fused_conv1" in t:
        return {"dram_bytes_per_step": t["dram_bytes_total_with_fused_conv1"],
                "vs_algorithmic": t.get("vs_algorithmic_with_fused_conv1"),
                "note": "conv1_fused_tc_kernel (its own ncu --set full capture, profiles/r02_conv1_fused.md) + the 11 "
                        "conv3x3_tc_kernel launches conv2_1..conv5_3 of one batch-32 step (per-layer table "
                        f"profiles/r02_conv_traffic.json / .md, {t.get('captured', 'ncu')}): ncu dram read+write"}
    return {"dram_bytes_per_step": t["dram_bytes_total"], "vs_algorithmic": t.get("vs_algorithmic"),
            "note": f"sum over the 12 conv3x3_tc_kernel launches of one step, ncu dram read+write, per-layer table in "
                    f"profiles/r02_conv_traffic.json / .md ({t.get('captured', 'ncu')})"}


def load_json_profile(name):
    p = os.path.join(ROOT, "profiles", name)
    return json.load(open(p)) if os.path.exists(p) else {}


def cpu_thread_candidates():
    cores = os.cpu_count() or 1
    cand = sorted({c for c in (32, 64, 128, cores) if c <= cores}) or [cores]
    return cand, cores


def cpu_reference_setup():
    from openibl_b200 import synth
    sd = synth.make_state_dict(seed=0, with_pca=True)
    return sd


def cpu_pick_threads(sd, probe_images=2):
    """Sweep the intra-op thread count on a small probe (after one warm-up pass): MKL/oneDNN convs on a 128-core
    box are often fastest well below the core count, and round 1's fixed 128 threads moved 3.7x box to box."""
    from oracle import ibl_oracle as O
    from openibl_b200 import synth
    x = synth.make_images(seed=1, batch=probe_images)
    cand, cores = cpu_thread_candidates()
    best, rates = None, {}
    with torch.no_grad():
        for t in cand:
            torch.set_num_threads(t)
            O.extract_descriptor(x[:1], sd)                 # warm-up at this thread count
            t0 = time.perf_counter()
            O.extract_descriptor(x, sd)
            rates[t] = probe_images / (time.perf_counter() - t0)
            if best is None or rates[t] > rates[best]:
                best = t
    torch.set_num_threads(best)
    return best, rates, cores


def cpu_reference_images_per_sec(n_images: int, sd=None):
    """Reference arithmetic on the host cores: oracle port of EmbedNetPCA.forward (evaluators.py:22-34 +
    netvlad.py:95-110), full warm-up pass, best thread count of the sweep."""
    from oracle import ibl_oracle as O
    from openibl_b200 import synth
    sd = sd or cpu_reference_setup()
    threads, rates, cores = cpu_pick_threads(sd)
    x = synth.make_images(seed=1, batch=n_images)
    with torch.no_grad():
        O.extract_descriptor(x, sd)                         # full warm-up pass (allocator, oneDNN primitives)
        t0 = time.perf_counter()
        O.extract_descriptor(x, sd)
        dt = time.perf_counter() - t0
    return n_images / dt, dt, threads, rates, cores


def cpu_reference_pairs_per_sec(nq: int, ndb: int):
    from oracle import ibl_oracle as O
    from openibl_b200 import synth
    q, db, _ = synth.make_gallery(ndb, nq, DIM)
    t0 = time.perf_counter()
    d = O.pairwise_distance(q, db).numpy()
    O.topk_from_distmat(d, TOPK)
    dt = time.perf_counter() - t0
    return nq * ndb / dt, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ibl_oracle as O
    from openibl_b200 import synth
    sd = cpu_reference_setup()                                 # parameters and inputs are built outside
    threads, rates, cores = cpu_pick_threads(sd)               # the timed region, as on the GPU arm
    # bounded sample of the batch-32 workload: >= 8 images per step unless K steps of that would run past ~5 min
    rate = rates[threads]
    per_step = 8
    if args.steps * per_step / rate > 300.0:
        per_step = max(2, int(300.0 * rate / max(args.steps, 1)))
    x = synth.make_images(seed=1, batch=per_step)
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 2))):
            O.extract_descriptor(x, sd)                        # full warm-up passes
        t0 = time.perf_counter()
        n = 0
        for _ in range(args.steps):
            O.extract_descriptor(x, sd)
            n += per_step
        dt = time.perf_counter() - t0
    val = n / dt
    pps, _ = cpu_reference_pairs_per_sec(400, NDB)
    line = {
        "impl": "reference", "metric": "images_per_sec_extraction", "value": val, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "batch-32 3x480x640 VGG16+NetVLAD+PCA(4096) extraction (configs[1])",
                   "sample": f"{per_step} images per step", "threads": threads,
                   "thread_sweep_images_per_s": {str(k): round(v, 3) for k, v in rates.items()}},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": threads, "host_cores": cores, "kind": "port",
                         "sample": f"{per_step} images/step x {args.steps} steps of the batch-32 workload, "
                                   f"best of thread sweep {sorted(rates)}"},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "retrieval": {"metric": "query_db_pairs_per_sec", "value": pps, "unit": "pairs/s",
                      "sample": f"400 x {NDB} x {DIM} pairwise_distance + top-{TOPK}"},
    }
    print(json.dumps(line), flush=True)


def gpu_eager_images_per_sec(xs, sd_dev, steps=3):
    """What stock PyTorch gets on the SAME B200 (SURVEY 2.1 'the bar', BASELINE.md 3.4): the reference forward as
    eager torch ops on CUDA tensors -- cuDNN convs (cudnn.benchmark=True as examples/test.py:80), cuBLAS GEMMs, ATen
    normalisations -- batch 32, same inputs and weights.  Two variants: fp32-strict (TF32 off; the arithmetic the
    1e-4 tolerance is stated against) and torch defaults (cuDNN convs may use TF32).  The NetVLAD aggregation is the
    oracle's einsum form, which is FASTER than the reference's literal [B,64,512,1200] temporary (netvlad.py:56-59)."""
    from oracle import ibl_oracle as O
    import torch.backends.cudnn as cudnn
    out = {}
    old = (cudnn.benchmark, cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    cudnn.benchmark = True
    try:
        for name, tf32 in (("fp32_strict", False), ("torch_default", None)):
            if tf32 is not None:
                cudnn.allow_tf32 = tf32
                torch.backends.cuda.matmul.allow_tf32 = tf32
            else:
                cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = True, False      # torch 2.11 defaults
            with torch.no_grad():
                for i in range(2):
                    O.extract_descriptor(xs[i % 2], sd_dev)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(steps):
                    O.extract_descriptor(xs[i % 2], sd_dev)
                e1.record()
                torch.cuda.synchronize()
            out[name] = {"value": BATCH * steps / (e0.elapsed_time(e1) / 1000.0), "unit": "images/s",
                         "ms_per_step": e0.elapsed_time(e1) / steps}
    finally:
        cudnn.benchmark, cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        torch.cuda.empty_cache()
    out["note"] = ("eager torch 2.11 ops (cuDNN/cuBLAS/ATen) through the oracle's functional forward, cudnn.benchmark=True, "
                   "batch 32, device-resident inputs; library kernels -- a baseline, not the product path")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--conv-mode", default="tc", choices=["tc", "simt"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager", action="store_true", help="skip the stock-PyTorch (cuDNN) leg")
    ap.add_argument("--no-strong", action="store_true", help="skip the 250k-image strong-scaling leg")
    ap.add_argument("--strong-db", type=int, default=250000)
    ap.add_argument("--strong-budget-s", type=float, default=240.0,
                    help="skip the strong-scaling leg if its projected extraction time exceeds this")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed extraction and retrieval steps to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the B200 engine, not to --impl reference")
        return run_reference(args)

    import torch.distributed as dist
    from openibl_b200 import synth
    from openibl_b200.engine import Engine, CONV_SIMT_FP32, CONV_TC_BF16X3

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng = Engine.get(local)
    eng.conv_mode = CONV_TC_BF16X3 if args.conv_mode == "tc" else CONV_SIMT_FP32
    sd = {k: v.to(dev) for k, v in synth.make_state_dict(seed=0, with_pca=True).items()}
    slots = synth.VGG16_CONV_SLOTS
    eng.set_vgg16([sd[f"base_model.base.{s}.weight"] for s in slots], [sd[f"base_model.base.{s}.bias"] for s in slots])
    eng.set_netvlad(sd["net_vlad.conv.weight"], sd["net_vlad.centroids"])
    eng.set_pca(sd["pca_layer.weight"], sd["pca_layer.bias"])

    # two distinct input batches (2 x 118 MB > L2) alternate between steps
    xs_host = [synth.make_images(seed=100 + 2 * rank + i, batch=BATCH).pin_memory() for i in range(2)]
    xs = [x.to(dev) for x in xs_host]
    out_host = torch.empty(BATCH, 4096).pin_memory()

    # ---- device-resident throughput -------------------------------------------------------
    for i in range(max(args.warmup, 3)):
        eng.extract(xs[i % 2], pca=True)
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        desc, _ = eng.extract(xs[i % 2], pca=True)
    e1.record()
    torch.cuda.synchronize()
    launches = eng.launch_count - l0
    dumped = {"descriptors": desc.cpu()}
    del desc
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    value = world * BATCH * args.steps / (ms_total / 1000.0)

    # ---- backbone alone (dominant kernel family) for the roofline ----------------------------
    feat = torch.empty(BATCH, 30, 40, 512, device=dev)
    from openibl_b200.engine import _ptr, _stream, check
    def backbone(x):
        check(eng.lib.ibl_vgg16_forward(eng.h, _ptr(x), BATCH, H, W, _ptr(feat), None, None, _stream(local)), "vgg")
    backbone(xs[0])
    torch.cuda.synchronize()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record()
    nb = max(3, min(args.steps, 10))
    for i in range(nb):
        backbone(xs[i % 2])
    b1.record()
    torch.cuda.synchronize()
    bb_ms = b0.elapsed_time(b1) / nb
    pk = peaks()
    ach = GFLOP_PER_IMAGE_BACKBONE * BATCH / bb_ms          # GFLOP/ms == TFLOP/s
    # the dominant kernel itself: conv3x3_tc_kernel, timed launch by launch (12 layers, CUDA events inside
    # the library on the launching stream, 3 repetitions each after a warm-up launch)
    import ctypes
    shapes, hh, ww = [], H, W
    for item in synth.VGG16_PLAN:
        if item == "P":
            hh, ww = hh // 2, ww // 2
        else:
            shapes.append((hh, ww, item[1], item[2]))
    conv_ms, conv_gflop = 0.0, 0.0
    fused1 = os.environ.get("IBL_CONV1_FUSED", "1") != "0"
    for li, (lh, lw, cin, cout) in enumerate(shapes):
        if li == 0 and not fused1:
            continue                      # conv1_1 alone (Cin = 3, output-write bound) is not part of the family
        if li == 1 and fused1:
            continue                      # conv1_2 is inside the fused conv1 kernel timed at li == 0
        msl = ctypes.c_float()
        if li == 0:                       # conv1_1 + conv1_2 + pool in ONE kernel: layer id 13, NCHW image input
            check(eng.lib.ibl_debug_time_layer(eng.h, 13, _ptr(xs[0]), BATCH, lh, lw, 0, 3, ctypes.byref(msl)), "time_layer")
            conv_gflop += 2.0 * BATCH * lh * lw * 9 * (3 * 64 + 64 * 64) / 1e9
        else:
            xin = torch.randn(BATCH, lh, lw, cin, device=dev).relu_()
            check(eng.lib.ibl_debug_time_layer(eng.h, li, _ptr(xin), BATCH, lh, lw, 0, 3, ctypes.byref(msl)), "time_layer")
            conv_gflop += 2.0 * BATCH * lh * lw * 9 * cin * cout / 1e9
            del xin
        conv_ms += msl.value
    ach_k = conv_gflop / conv_ms
    conv_traffic = load_conv_traffic()
    roofline = {"bound": "tensor",
                "kernel": ("conv1_fused_tc_kernel (conv1_1+conv1_2+pool) + conv3x3_tc_kernel x 11 (conv2_1..conv5_3): 12 launches, "
                           "tcgen05 implicit GEMM, bf16x3") if fused1 else
                          "conv3x3_tc_kernel (12 launches: conv1_2..conv5_3, tcgen05 implicit GEMM, bf16x3)",
                "achieved": ach_k, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": ach_k / pk["bf16_tflops_sustained"],
                "traffic": conv_traffic.get("dram_bytes_per_step"), "traffic_note": conv_traffic.get("note"),
                "traffic_vs_algorithmic": conv_traffic.get("vs_algorithmic"),
                "peak_source": pk["src"] + " bf16 sustained (cuBLAS)",
                "note": "achieved = algorithmic fp32-grade FLOPs / sum of the 12 launch durations; the bf16x3 split issues "
                        "3 MMA passes per product, so the tensor pipe executes 3x the algorithmic figure (mma_issue_frac)",
                "ms_per_launch_group": conv_ms, "mma_issue_frac": 3 * ach_k / pk["bf16_tflops_sustained"],
                "backbone_13_launches": {"ms": bb_ms, "achieved": ach, "frac": ach / pk["bf16_tflops_sustained"]}}

    # ---- end to end through host buffers -----------------------------------------------------
    # (a) the blocking call: H2D + path + D2H + sync per step (ibl_extract_host)
    for i in range(2):
        eng.extract_host(xs_host[i % 2], out_host, pca=True)
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for i in range(args.steps):
        eng.extract_host(xs_host[i % 2], out_host, pca=True)
    g1.record()
    torch.cuda.synchronize()
    e2e_ms = torch.tensor([g0.elapsed_time(g1)], device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_blocking_val = world * BATCH * args.steps / (float(e2e_ms.item()) / 1000.0)
    # (b) the two-slot pipelined call (ibl_extract_host_submit / _wait): every step still copies ITS inputs host->device
    # and ITS descriptors device->host inside the timed region; the copy of step i+1 runs under the compute of step i
    outs_host = [torch.empty(BATCH, 4096).pin_memory() for _ in range(2)]
    for _ in eng.extract_host_stream(((xs_host[i % 2], outs_host[i % 2]) for i in range(3)), pca=True):
        pass
    barrier()
    t_wall0 = time.perf_counter()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    n_done = 0
    for _ in eng.extract_host_stream(((xs_host[i % 2], outs_host[i % 2]) for i in range(args.steps)), pca=True):
        n_done += 1
    p1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t_wall0) * 1000.0
    assert n_done == args.steps
    pipe_ms = torch.tensor([max(p0.elapsed_time(p1), wall_ms)], device=dev)     # device time, never less than the host's wall clock
    if world > 1:
        dist.all_reduce(pipe_ms, op=dist.ReduceOp.MAX)
    e2e_val = world * BATCH * args.steps / (float(pipe_ms.item()) / 1000.0)

    # ---- the same from decoded uint8 HWC images (ToTensor + Normalize on the device) -------------
    from openibl_b200.utils.data import _MEAN, _STD
    gu = torch.Generator().manual_seed(11 + rank)
    xs_u8 = [torch.randint(0, 256, (BATCH, H, W, 3), dtype=torch.uint8, generator=gu).pin_memory() for _ in range(2)]
    for i in range(2):
        eng.extract_host_u8(xs_u8[i % 2], out_host, _MEAN, _STD, pca=True)
    barrier()
    u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    u0.record()
    for i in range(args.steps):
        eng.extract_host_u8(xs_u8[i % 2], out_host, _MEAN, _STD, pca=True)
    u1.record()
    torch.cuda.synchronize()
    u8_ms = torch.tensor([u0.elapsed_time(u1)], device=dev)
    if world > 1:
        dist.all_reduce(u8_ms, op=dist.ReduceOp.MAX)
    e2e_u8_val = world * BATCH * args.steps / (float(u8_ms.item()) / 1000.0)
    del xs_u8

    # ---- retrieval: 6.8k x (10k per rank) sharded distance + top-k + all-gather merge ----------
    from openibl_b200.evaluators import sharded_topk
    q, db, gt = synth.make_gallery(NDB, NQ, DIM, seed_db=2 + rank)
    qd, dbd = q.to(dev), db.to(dev)
    for _ in range(2):
        sharded_topk(qd, dbd, TOPK, idx_base=rank * NDB, n_valid=NDB)
    barrier()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    rsteps = 3
    for _ in range(rsteps):
        top_d, top_i = sharded_topk(qd, dbd, TOPK, idx_base=rank * NDB, n_valid=NDB)
    r1.record()
    torch.cuda.synchronize()
    dumped["retrieval_topk_dist"], dumped["retrieval_topk_idx"] = top_d.cpu(), top_i.cpu().double()
    del top_d, top_i
    r_ms = torch.tensor([r0.elapsed_time(r1) / rsteps], device=dev)
    if world > 1:
        dist.all_reduce(r_ms, op=dist.ReduceOp.MAX)
    pairs = NQ * NDB * world / (float(r_ms.item()) / 1000.0)

    # ---- stock PyTorch on the same GPU (cuDNN / cuBLAS eager): rank 0 only -----------------------
    eager = None
    if rank == 0 and not args.no_eager:
        try:
            eager = gpu_eager_images_per_sec(xs, sd)
        except Exception as exc:   # a baseline leg must never take the bench line down
            eager = {"unavailable": repr(exc)[:200]}
    barrier()

    # ---- configs[3]: 250k-image gallery sharded over the ranks, strong scaling ---------------------
    strong = None
    if not args.no_strong:
        from openibl_b200 import gallery
        proj = args.strong_db / max(value, 1.0)          # seconds of extraction at the rate just measured (all ranks)
        if proj > args.strong_budget_s:
            strong = {"skipped": f"projected extraction time {proj:.0f} s exceeds --strong-budget-s {args.strong_budget_s:.0f}"}
        else:
            # PCA bias = -W.mean of a database sample, as a PCA fit sets it (ibl/pca.py:86-90): without the centring a
            # random-init trunk's descriptors are ~1e-5 apart and the ranking is decided by rounding noise
            gallery.center_pca(eng, sd["pca_layer.weight"], H, W, BATCH)
            # warm-up outside the timed region: allocations, NCCL communicator and its first-call setup
            gallery.run(eng, 2 * BATCH * world, 64, H, W, BATCH, check_exact=False)
            strong = gallery.run(eng, args.strong_db, NQ, H, W, BATCH, check_exact=False)
            strong["guard_flagged_queries_rank0"] = eng.dist_flagged()
            eng.set_pca(sd["pca_layer.weight"], sd["pca_layer.bias"], force=True)
            strong["note"] = ("same 250k-image gallery whatever N (images seeded by global index): topk_index_hash and "
                              "recalls must be equal across N; total_s is the strong-scaling time (max over ranks)")

    if rank == 0:
        pk_burst = pk["bf16_tflops"]
        r_alg = 2.0 * NQ * NDB * DIM * world / (float(r_ms.item()) / 1000.0) / 1e12
        dist_prof = load_json_profile("r02_dist_tensor_pipe.json")
        line = {
            "metric": "images_per_sec_extraction", "value": value, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (bf16x3 split on tcgen05, fp32 accumulate)" if args.conv_mode == "tc" else "f32",
            "data": "synthetic",
            "config": {"workload": "batch-32 3x480x640 VGG16+NetVLAD+PCA(4096) extraction per GPU (configs[1])",
                       "global_batch": BATCH * world, "l2": "two alternating 118 MB input batches; 2.5 GB of "
                       "inter-layer activations per step evict L2", "parallelism": f"dp{world}",
                       "conv_mode": args.conv_mode},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "e2e": {"value": e2e_val, "unit": "images/s",
                    "h2d_bytes_per_step": BATCH * 3 * H * W * 4, "d2h_bytes_per_step": BATCH * 4096 * 4,
                    "api": "Engine.extract_host_stream (ibl_extract_host_submit/_wait, two slots): pinned fp32 host batches in, "
                           "pinned descriptors out, every step's H2D and D2H inside the timed region",
                    "blocking_call_value": e2e_blocking_val},
            "e2e_u8": {"value": e2e_u8_val, "unit": "images/s", "h2d_bytes_per_step": BATCH * 3 * H * W,
                       "d2h_bytes_per_step": BATCH * 4096 * 4,
                       "note": "same path fed with decoded uint8 HWC images; ToTensor+Normalize "
                               "(ibl/utils/data/__init__.py:37-42) runs on the device"},
            "retrieval": {"metric": "query_db_pairs_per_sec", "value": pairs, "unit": "pairs/s",
                          "workload": f"{NQ} q x {NDB} db/GPU x {DIM}-d, top-{TOPK}, sharded + all-gather merge",
                          "ms": float(r_ms.item()), "algorithmic_tflops": r_alg,
                          "roofline": {"bound": "tensor", "achieved": r_alg / world, "peak": pk_burst, "unit": "TFLOP/s",
                                       "frac": r_alg / world / pk_burst,
                                       "peak_source": pk["src"] + " bf16 burst (cuBLAS), kernel timed alone",
                                       "tensor_pipe_active_pct": dist_prof.get("tensor_pipe_active_pct"),
                                       "tensor_pipe_source": dist_prof.get("source"),
                                       "note": "achieved = 2*m*n*d algorithmic FLOP of the whole call (planes + screening "
                                               "GEMM + merge + exact re-scoring) per GPU / its CUDA-event time"}},
        }
        if eager is not None:
            line["gpu_eager"] = eager
        if strong is not None:
            line["strong_250k"] = strong
        if not args.no_cpu_baseline and world == 1:
            v, dt, threads, rates, cores = cpu_reference_images_per_sec(8)
            line["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": threads, "host_cores": cores, "kind": "port",
                                    "thread_sweep_images_per_s": {str(k): round(r, 3) for k, r in rates.items()},
                                    "sample": f"8 of the 32 images of one step after a full warm-up pass, oracle "
                                              f"EmbedNetPCA forward, {dt:.1f} s, best thread count of the sweep"}
        if args.dump_outputs:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, t in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), t.numpy())
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
