#!/usr/bin/env python
"""bench.py - CVAE-GAN training throughput (train samples/s) on synthetic Car-Hacking-shaped data.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU implementation (oracle port)
    python bench.py --steps K --dump-outputs DIR             # also write what the last timed step computed, as .npy

Workload (BASELINE.json configs[1]; SURVEY.md 8d "C2"): F=10 features (CAN ID, DLC, 8 data bytes), K=5
classes, Z=128, fp32, batch 4096 rows PER GPU (weak scaling: global batch 4096*N).  One bench "step" is
ONE LABEL VISIT of the reference's training loop (cvae_gan.py:102-216): 5 critic + 5 classifier +
3 encoder/generator optimiser steps, each on a freshly sampled batch => 13 * batch train samples.
metric = train samples/s = 13 * global_batch * steps / time   (BASELINE.md section 3).

Timed region of `value`: class tables resident in HBM, row sampling (_get_target_samples) on the
device, 13 optimiser steps per visit, nothing read back.  `e2e`: the same visits driven through the
public step API with each step's batch copied from PINNED HOST memory (H2D) and each step's losses
copied back (D2H) inside the timed region.  Inputs are larger than L2: the class tables total 200 MB
and every step gathers random rows from them.
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
sys.path.insert(0, ROOT)

F_, K_, Z_ = 10, 5, 128
BATCH_PER_GPU = int(os.environ.get("CVG_BENCH_BATCH", "4096"))   # 4096 = BASELINE.json configs[1]; env override is a probe only
ROWS_PER_CLASS = 1_000_000          # 5 * 1e6 * 40 B = 200 MB > 126 MB L2
D_LOOP, C_LOOP, G_LOOP = 5, 5, 3    # gan_config.py:7,10,13
OPT_STEPS = D_LOOP + C_LOOP + G_LOOP
# minimal algorithmic work per train sample, F=10 K=5 (SURVEY.md 8d / BASELINE.md section 3)
FLOP_PER_SAMPLE = 873_945
WIDE_HIDDEN = (1024, 512, 256)      # BASELINE.json configs[4] / SURVEY 8(d) C5: the widened model (fp32 here; no bf16 path)


def flop_per_train_sample(F, K, Z, hidden=None):
    """SURVEY.md 8(d) accounting (minimal algorithmic work, MACs per batch row) for any layer widths: forward MACs of every
    pass, backward = weight gradient + input gradient per layer, minus the input gradients nobody needs (first layers of the
    trained networks; the critic's / classifier's weight gradients in the encoder/generator step).  2 FLOP per MAC, 13
    optimiser steps of one row each per label visit.  flop_per_train_sample(10, 5, 128) = 873 945 (the SURVEY figure)."""
    def widths(tin, fixed3):
        return tuple(hidden) if hidden else (max(256, tin), max(128, tin // 2), 64 if fixed3 else max(64, tin // 4))

    def macs(dims):
        return sum(a * b for a, b in zip(dims[:-1], dims[1:]))
    eh, gh, dh, ch = widths(F + K, False), widths(Z + K, False), widths(F + K, True), widths(F, True)
    mE = macs((F + K, *eh)) + eh[2] * 2 * Z
    mG = macs((Z + K, *gh, F))
    mD = macs((F + K, *dh, 1))
    mC = macs((F, *ch, K))
    d_step = mG + 2 * mD + 2 * (2 * mD - (F + K) * dh[0])
    c_step = mG + 2 * mC + 2 * (2 * mC - F * ch[0])
    g_bwd = mD + mC + (4 * mG - (Z + K) * gh[0] - K * gh[0]) + (2 * mE - (F + K) * eh[0])
    g_step = mE + 2 * mG + mD + mC + g_bwd
    return 2.0 * (D_LOOP * d_step + C_LOOP * c_step + G_LOOP * g_step) / OPT_STEPS



def ncu_traffic():
    """DRAM bytes per launch from the committed ncu captures (profiles/r1_traffic.json), or {}."""
    p = os.path.join(ROOT, "profiles", "r1_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synth_class_tables(device, rows_per_class, seed=0):
    """Car-Hacking-shaped rows in [0,1]: per class a centre + spread (make_blobs -> minmax_scale, utils.py:56-66)."""
    import torch
    g = torch.Generator(device="cpu").manual_seed(seed)
    tabs = []
    for k in range(K_):
        c = torch.rand(F_, generator=g)
        gd = torch.Generator(device=device).manual_seed(seed * 100 + k)
        t = (c.to(device) + 0.08 * torch.randn(rows_per_class, F_, generator=gd, device=device)).clamp_(0, 1)
        tabs.append(t.contiguous())
    return tabs


# ---------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's CPU path, timed on the host cores
# ---------------------------------------------------------------------------------------------------------
def time_cpu_port(visits: int, warm: int, batch: int, threads: int, rows_per_class=20000, hidden=None):
    """Label visits of the reference algorithm (oracle port, torch CPU ops, torch RNG like the reference)."""
    import torch
    from oracle import cvae_gan_oracle as O
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(0)
    cfg = O.OracleConfig(batch_size=batch, hidden=hidden)
    orc = O.OracleCVAEGAN(F_, K_, cfg).init_like_reference(g)
    orc.make_optimizers()
    xs = [(torch.rand(F_, generator=g) + 0.08 * torch.randn(rows_per_class, F_, generator=g)).clamp(0, 1) for _ in range(K_)]
    for k in range(K_):
        orc.samples[k] = xs[k]
    noise = O.TorchNoise()

    def visit(label):
        for _ in range(D_LOOP):
            orc.step_d(orc.get_target_samples(label, batch, noise), label, noise)
        for _ in range(C_LOOP):
            orc.step_c(orc.get_target_samples(label, batch, noise), label, noise)
        for _ in range(G_LOOP):
            orc.step_g(orc.get_target_samples(label, batch, noise), label, noise, 0.25)

    for i in range(warm):
        visit(i % K_)
    t0 = time.perf_counter()
    for i in range(visits):
        visit(i % K_)
    dt = time.perf_counter() - t0
    return OPT_STEPS * batch * visits / dt, dt / visits


def time_cpu_filter_port(threads: int, budget_s: float = 6.0):
    """The reference's generation + classifier-confidence filter on the host cores (oracle port), two ways (SURVEY 8d):
    `generate_qualified_samples` as written (chunks of <= 10 rows, cvae_gan.py:347-378) and one vectorised
    generate -> classify -> filter call.  Returns generated rows/s of both."""
    import torch
    from oracle import cvae_gan_oracle as O
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    orc = O.OracleCVAEGAN(F_, K_, O.OracleConfig(batch_size=64)).init_like_reference(g)
    for k in orc.training:
        orc.training[k] = False                       # after fit() every network is in eval mode (cvae_gan.py:233-236)
    torch.manual_seed(0)
    with torch.no_grad():
        probe = orc.classify_eval(orc.generate_samples(0, 2000)).argmax(1)
    label = int(torch.bincount(probe, minlength=K_).argmax())   # a label this (untrained) classifier does accept at thr 0

    class Counting(O.TorchNoise):
        rows = 0

        def randn(self, rows, cols, tag=""):
            Counting.rows += rows
            return super().randn(rows, cols, tag)

    noise = Counting()
    t0 = time.perf_counter()
    asked = 0
    while time.perf_counter() - t0 < budget_s / 2:
        orc.generate_qualified_samples(label, 2000, thr=0.0, noise=noise)
        asked += 2000
    dt_chunk = time.perf_counter() - t0
    chunked = Counting.rows / dt_chunk
    n_vec = 200_000
    z = torch.randn(n_vec, Z_)
    t0 = time.perf_counter()
    reps = 0
    while time.perf_counter() - t0 < budget_s / 2:
        orc.generate_filter_stream(label, z, 0.0)
        reps += 1
    vec = reps * n_vec / (time.perf_counter() - t0)
    return {"chunked_generated_rows_per_s": chunked, "vectorised_generated_rows_per_s": vec, "label": label, "threshold": 0.0,
            "sample": f"oracle port on {threads} threads: generate_qualified_samples in chunks of 10 for {dt_chunk:.1f} s "
                      f"({Counting.rows} rows), and {reps} vectorised passes over {n_vec} rows"}


WORKLOAD = ("CVAE-GAN training, Car-Hacking shape F=10 K=5 Z=128, fp32, batch 4096 per GPU "
            "(BASELINE.json configs[1]); step = one label visit = 5 D + 5 C + 3 E/G optimiser steps")
REF_BUDGET_S = float(os.environ.get("CVG_BENCH_REF_BUDGET_S", "150"))


def run_reference(args):
    """The reference's CPU implementation of the path (oracle port of src/cvae_gan.py: /root/reference does not exist on the
    GPU box) on all host cores, same workload / metric / steps as our arm.  --steps and --warmup are honoured; only when the
    run would exceed REF_BUDGET_S seconds are the steps cut, and the line then says so (steps_requested)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    batch = BATCH_PER_GPU * args.gpus
    warm = max(args.warmup, 0)
    _, per0 = time_cpu_port(1, 1, batch, cores)                     # one visit to size the run
    visits = max(1, min(args.steps, int(REF_BUDGET_S / max(per0, 1e-3)) - warm))
    warm = min(warm, max(0, int(0.25 * REF_BUDGET_S / max(per0, 1e-3))))
    val, per = time_cpu_port(visits, warm, batch, cores)
    line = {
        "impl": "reference", "metric": "train_samples_per_s", "value": val, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": visits, "warmup": warm, "ms_per_step": per * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": batch, "batch_per_gpu": BATCH_PER_GPU, "opt_steps_per_step": OPT_STEPS,
                   "device": "host CPU", "torch_threads": cores, "steps_requested": args.steps, "warmup_requested": args.warmup,
                   "time_budget_s": REF_BUDGET_S},
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"{visits} label visits ({visits * OPT_STEPS} optimiser steps) at batch {batch}, "
                                   "oracle port of src/cvae_gan.py on torch CPU ops"},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, eng, loss):
    """What the timed label visits hand back to a caller, as float32 .npy files (about 1 MB in all): `losses.npy`, the
    13 x 4 losses of the last visit, and `<network>.<state_dict key>.npy` for every tensor of the four networks after it.
    The inputs depend only on the command-line arguments.  Weight and LayerNorm-affine gradients are summed exactly (fixed
    point, gemm_dw_kernel / ln_bwd_kernel), so the order the GPU adds them in cannot change them; BatchNorm statistics and
    loss sums still use double-precision atomics, whose order can move the last bit of a double before it is rounded to
    float32.  Measured on one B200 (1000 W limit): two runs with the same arguments wrote bit-identical files at --steps 1,
    50 and 100."""
    import numpy as np
    from cvae_gan_b200._lib import NET_NAMES
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "losses.npy"), loss.cpu().numpy())
    for net, name in enumerate(NET_NAMES):
        for key, t in eng.export_state(net).items():
            np.save(os.path.join(out_dir, f"{name}.{key}.npy"), t.cpu().numpy())


def _finish(eng, world):
    """Leave the process without running communicator destructors: with several ranks, tearing down the library's NCCL
    communicator and torch's process group in arbitrary order has been seen to block for minutes after the result line
    was printed.  Every rank has finished its GPU work here (barrier), so exiting is safe."""
    import torch
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    eng.close()


# ---------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from cvae_gan_b200.engine import Engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B = BATCH_PER_GPU
    Bg = B * world
    eng = Engine(F_, K_, Z_, max_batch=B, world_size=world, rank=rank)
    # reference-distributed random-init weights (no checkpoints offline)
    from cvae_gan_b200 import models
    torch.manual_seed(0)
    mods = [models.CVAEGANEncoderModel(F_, K_, Z_), models.CVAEGANGeneratorModel(Z_, K_, F_),
            models.CVAEGANDiscriminatorModel(F_, K_), models.CVAEGANClassifierModel(F_, K_)]
    for net, m in enumerate(mods):
        eng.load_state(net, m.state_dict())
    if args.only_filter:
        r = run_filter_leg(eng, dev, world, rank, peaks())
        if rank == 0:
            print(json.dumps(r), flush=True)
        _finish(eng, world)
        return
    dp_par = None
    if world > 1:
        # data-parallel correctness BEFORE anything is timed: one D / C / G step on K=4 imbalanced data against a
        # single-GPU run on the global batch (tools/dp_parity.py); a failing check fails the run
        from tools.dp_parity import run_dp_parity
        dp_par = run_dp_parity(world, rank, dev, B)
        if not dp_par["ok"]:
            if rank == 0:
                print(json.dumps({"error": "dp_parity failed", "dp_parity": dp_par}), flush=True)
            dist.barrier()
            os._exit(3)
    tabs = synth_class_tables(dev, ROWS_PER_CLASS, seed=0)
    seed = 1234
    loss = torch.zeros(OPT_STEPS, 4, device=dev)
    LOOPS = (D_LOOP, C_LOOP, G_LOOP)
    if args.quick and os.environ.get("CVG_BENCH_LOOPS"):      # diagnostics: time one kind of step, e.g. "5,0,0"
        LOOPS = tuple(int(v) for v in os.environ["CVG_BENCH_LOOPS"].split(","))
    eng.ctl_set(seed=seed, counter=0, lambda_class=0.25)

    def visit_eager(label):
        eng.visit(label, Bg, class_rows=tabs[label], loops=LOOPS, loss_out=loss)

    # launches of one label visit (the graphs replay exactly these)
    l0 = eng.launch_count()
    visit_eager(0)
    launches_per_visit = eng.launch_count() - l0
    torch.cuda.synchronize()

    # value: class tables resident in HBM, rows drawn on the device, one CUDA graph per label
    graphs = {}
    for label in range(K_):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            # --quick only (diagnostics): CVG_BENCH_VISIT_FLAGS=2 times the visit with per-rank BatchNorm sums
            eng.visit(label, Bg, class_rows=tabs[label], loops=LOOPS, loss_out=loss,
                      flags=int(os.environ.get("CVG_BENCH_VISIT_FLAGS", "0")) if args.quick else 0)
        graphs[label] = g

    def visit_resident(label):
        graphs[label].replay()

    # e2e: the 13 batches of a visit come from PINNED HOST memory (one H2D copy per visit into a staging
    # buffer the graph reads), the 13 x 4 losses go back to pinned host memory, then the host waits
    ring = 8
    gcpu = torch.Generator().manual_seed(rank + 1)
    host_batches = torch.empty(ring, OPT_STEPS, B, F_).pin_memory()
    for r in range(ring):
        idx = torch.randint(0, ROWS_PER_CLASS, (OPT_STEPS * B,), generator=gcpu)
        host_batches[r].copy_(tabs[r % K_][idx.to(dev)].view(OPT_STEPS, B, F_).cpu())
    host_loss = torch.zeros(OPT_STEPS, 4).pin_memory()
    x_stage = torch.empty(OPT_STEPS, B, F_, device=dev)
    graphs_e2e = {}
    for label in range(K_):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            eng.visit(label, Bg, x_batches=x_stage, loops=LOOPS, loss_out=loss)
        graphs_e2e[label] = g
    slot = [0]

    def visit_e2e(label):
        x_stage.copy_(host_batches[slot[0] % ring], non_blocking=True)
        slot[0] += 1
        graphs_e2e[label].replay()
        host_loss.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()      # the caller reads the losses of this visit

    def timed(fn, steps, warm):
        for i in range(warm):
            fn(i % K_)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i % K_)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    warm = args.warmup if args.quick else max(args.warmup, 3)
    if args.quick:
        ms = timed(visit_resident, args.steps, warm)
        if rank == 0:
            print(json.dumps({"quick": True, "ms_per_step": ms / args.steps, "launches": eng.launch_count()}), flush=True)
        _finish(eng, world)
        return
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms = timed(visit_resident, args.steps, warm)
    launches = launches_per_visit * args.steps
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, loss)     # before the e2e visits below overwrite losses and weights
    ms_e2e = timed(visit_e2e, args.steps, 1)
    value = OPT_STEPS * Bg * args.steps / (ms * 1e-3)
    e2e = OPT_STEPS * Bg * args.steps / (ms_e2e * 1e-3)
    final_losses = loss.tolist()
    ok = all(all(v == v and abs(v) < 1e6 for v in row) for row in final_losses)

    # ---- roofline of the dominant kernel class: every GEMM launch of two EAGER visits is bracketed by CUDA events on its
    # stream; the share is taken against the wall time of those same two eager visits (events around them) ----
    pk = peaks()
    eng.profile(True)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for i in range(2):
        visit_eager(i % K_)
    pe1.record()
    torch.cuda.synchronize()
    prof_wall_ms = pe0.elapsed_time(pe1)
    prof = eng.profile_read()
    eng.profile(False)
    top = max(prof, key=lambda k: prof[k][2])
    n_l, fl, t_ms = prof[top]
    achieved = fl / (t_ms * 1e-3) / 1e12 if t_ms > 0 else 0.0
    total_gemm_ms = sum(v[2] for v in prof.values())
    FP32_SIMT_NOMINAL = 148 * 128 * 2 * 1.965e9 / 1e12      # 74.5 TFLOP/s: 128 FMA lanes per SM at the maximum SM clock
    roofline = {
        "bound": "tensor", "kernel": top, "achieved": achieved, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
        "frac": achieved / pk["bf16_tflops_sustained"], "traffic": ncu_traffic().get(top, {}).get("bytes"), "peak_source": pk["source"] + " bf16 dense (sustained)",
        "pipe": "fp32 FFMA (CUDA cores): the default training executor; the tensor-pipe executor is reported in train_program",
        "frac_of_fp32_simt_nominal": achieved / FP32_SIMT_NOMINAL, "fp32_simt_nominal_tflops": FP32_SIMT_NOMINAL,
        "launches_profiled": n_l, "avg_launch_us": 1e3 * t_ms / max(n_l, 1),
        "gemm_share_of_eager_step": total_gemm_ms / prof_wall_ms, "eager_ms_per_step": prof_wall_ms / 2,
        "per_class": {k: {"launches": v[0], "tflops": (v[1] / (v[2] * 1e-3) / 1e12) if v[2] > 0 else 0.0, "ms": v[2]}
                      for k, v in prof.items()},
        "whole_step_tflops": value * FLOP_PER_SAMPLE / 1e12,
        "whole_step_frac": value * FLOP_PER_SAMPLE / 1e12 / pk["bf16_tflops_sustained"],
    }

    # ---- the tensor-pipe training executor (mega.cuh): the same visits as ONE persistent tcgen05 kernel each ----
    train_program = None
    if eng.debug_get("mk_supported"):
        eng.debug_set("train_mode", 1)
        try:
            l0 = eng.launch_count()
            visit_eager(0)                              # also allocates the program buffers outside stream capture
            prog_launches = eng.launch_count() - l0
            prog_ops = eng.debug_get("mk_last_nops")
            torch.cuda.synchronize()
            pg = {}
            for label in range(K_):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    eng.visit(label, Bg, class_rows=tabs[label], loops=LOOPS, loss_out=loss)
                pg[label] = g
            k_prog = args.steps
            ms_p = timed(lambda lab: pg[lab].replay(), k_prog, 3)
            train_program = {
                "ms_per_step": ms_p / k_prog, "value": OPT_STEPS * Bg * k_prog / (ms_p * 1e-3), "unit": "samples/s", "steps": k_prog,
                "gpu_launches_per_step": prog_launches, "ops_per_step": prog_ops,
                "kernel": "cvg::mk::step_program_kernel: one persistent cooperative kernel per label visit; every GEMM on "
                          "tcgen05.mma kind::tf32 (3xTF32), weights and activation rows streamed by TMA bulk copies, TMEM "
                          "accumulators, grid barriers instead of kernel boundaries, deterministic weight-gradient reduction",
                "whole_step_tflops": OPT_STEPS * Bg * k_prog / (ms_p * 1e-3) * FLOP_PER_SAMPLE / 1e12,
                "select": "CVG_TRAIN_MODE=mk (the FFMA executor is the default because it is faster at this batch size)",
            }
            del pg
        finally:
            eng.debug_set("train_mode", 0)

    # ---- BASELINE.json configs[4] (SURVEY 8d C5), single GPU, fp32: the widened model (hidden 1024 / 512 / 256 in all four
    # networks, CvgConfig.hidden) through the same label visits.  Informative leg: never lose the bench line over it. ----
    train_wide = None
    if world == 1 and not args.no_wide:
        try:
            train_wide = run_wide_leg(dev, tabs, timed, pk, args.steps)
        except Exception as ex:
            train_wide = {"error": str(ex)[:300]}

    # ---- the drop-in surface itself: CVAEGAN.fit(TrDataset()) + generate_qualified_samples (N = 1 only) ----
    e2e_fit = None
    if world == 1 and not args.no_fit:
        e2e_fit = run_fit_leg(dev)

    filt = None if args.no_filter else run_filter_leg(eng, dev, world, rank, pk)

    if rank == 0:
        cores = os.cpu_count() or 1
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            v8, _ = time_cpu_port(2, 1, BATCH_PER_GPU, cores)
            cpu = {"value": v8, "unit": "samples/s", "cores": cores, "kind": "port",
                   "sample": f"2 label visits (26 optimiser steps) at batch {BATCH_PER_GPU}, oracle port of src/cvae_gan.py, "
                             f"torch CPU ops, {cores} threads"}
        line = {
            "metric": "train_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "global_batch": Bg, "batch_per_gpu": B, "opt_steps_per_step": OPT_STEPS,
                       "launch": "one CUDA graph per label visit", "parallelism": f"dp{world}",
                       "exchange": ("none" if world == 1 else ("nvlink peer-memory LL all-reduce" if getattr(eng, "nvl", False) else "nccl")), "l2": "inputs larger than L2: 200 MB class tables, random row gather per step",
                       "losses_finite": ok},
            "e2e": {"value": e2e, "unit": "samples/s", "h2d_bytes_per_step": OPT_STEPS * B * F_ * 4,
                    "d2h_bytes_per_step": OPT_STEPS * 16, "ms_per_step": ms_e2e / args.steps,
                    "api": "cvg_visit with host-supplied batches: pinned H2D of the visit's 13 batches, graph replay, "
                           "pinned D2H of the 13 x 4 losses, host sync"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
        }
        if train_program:
            line["train_program"] = train_program
        if e2e_fit:
            line["e2e_fit"] = e2e_fit
        if train_wide:
            if cpu and "value" in train_wide:
                try:      # the same widened label visit on the host cores (oracle port with OracleConfig.hidden): 1 visit, no warm-up
                    vw, sw = time_cpu_port(1, 0, BATCH_PER_GPU, cores, hidden=WIDE_HIDDEN)
                    train_wide["cpu_baseline"] = {"value": vw, "unit": "samples/s", "cores": cores, "kind": "port",
                                                  "sample": f"1 label visit at batch {BATCH_PER_GPU}, {sw:.1f} s", "ratio": train_wide["value"] / vw}
                except Exception as ex:
                    train_wide["cpu_baseline"] = {"error": str(ex)[:200]}
            line["train_wide"] = train_wide
        if dp_par:
            line["dp_parity"] = dp_par
        if cpu:
            try:
                cpu["filter"] = time_cpu_filter_port(cores)
            except Exception as ex:          # the baseline is informative; never lose the bench line over it
                cpu["filter"] = {"error": str(ex)[:200]}
            line["cpu_baseline"] = cpu
        if filt:
            line["filter"] = filt
        print(json.dumps(line), flush=True)
    _finish(eng, world)



# ---------------------------------------------------------------------------------------------------------
# the widened model of BASELINE.json configs[4] on one GPU (fp32; the reference cannot express these widths)
# ---------------------------------------------------------------------------------------------------------
def run_wide_leg(dev, tabs, timed, pk, steps):
    import torch
    from cvae_gan_b200 import models
    from cvae_gan_b200.engine import Engine
    B = BATCH_PER_GPU
    eng = Engine(F_, K_, Z_, max_batch=B, hidden=WIDE_HIDDEN)
    try:
        torch.manual_seed(0)
        mods = [models.CVAEGANEncoderModel(F_, K_, Z_, hidden=WIDE_HIDDEN), models.CVAEGANGeneratorModel(Z_, K_, F_, hidden=WIDE_HIDDEN),
                models.CVAEGANDiscriminatorModel(F_, K_, hidden=WIDE_HIDDEN), models.CVAEGANClassifierModel(F_, K_, hidden=WIDE_HIDDEN)]
        for net, m in enumerate(mods):
            eng.load_state(net, m.state_dict())
        n_param = sum(int(p.numel()) for m in mods for p in m.parameters())
        loss = torch.zeros(OPT_STEPS, 4, device=dev)
        eng.ctl_set(seed=4321, counter=0, lambda_class=0.25)
        l0 = eng.launch_count()
        eng.visit(0, B, class_rows=tabs[0], loops=(D_LOOP, C_LOOP, G_LOOP), loss_out=loss)
        launches = eng.launch_count() - l0
        torch.cuda.synchronize()
        graphs = {}
        for label in range(K_):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                eng.visit(label, B, class_rows=tabs[label], loops=(D_LOOP, C_LOOP, G_LOOP), loss_out=loss)
            graphs[label] = g
        ms = timed(lambda lab: graphs[lab].replay(), steps, 3)
        fin = loss.tolist()
        value = OPT_STEPS * B * steps / (ms * 1e-3)
        flop = flop_per_train_sample(F_, K_, Z_, WIDE_HIDDEN)
        tf = value * flop / 1e12
        simt = 148 * 128 * 2 * 1.965e9 / 1e12
        del graphs
        return {"workload": f"widened CVAE-GAN, hidden {WIDE_HIDDEN} in all four networks, F={F_} K={K_} Z={Z_}, fp32 (NOT the bf16 "
                            f"variant BASELINE.json configs[4] names: no bf16 path is built), batch {B}, 1 GPU; same label visits",
                "value": value, "unit": "samples/s", "ms_per_step": ms / steps, "steps": steps, "parameters": n_param,
                "gpu_launches_per_step": launches, "flop_per_sample": flop, "whole_step_tflops": tf,
                "frac_of_fp32_simt_nominal": tf / simt, "frac_of_bf16_sustained": tf / pk["bf16_tflops_sustained"],
                "executor": "stand-alone fp32 FFMA layer kernels (the tcgen05 executors cover widths <= 256)",
                "losses_finite": all(all(v == v and abs(v) < 1e6 for v in row) for row in fin)}
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------------------
# the drop-in surface: CVAEGAN().fit(TrDataset()) and generate_qualified_samples, timed by the host clock
# ---------------------------------------------------------------------------------------------------------
def run_fit_leg(dev, epochs=6, rows_per_class=20000):
    """What a user of the reference calls (scripts/train_cvae_gan.py:47-66): set the dataset / config globals, construct
    CVAEGAN(), fit(TrDataset()), then top up a class with generate_qualified_samples.  The timed fit includes everything
    fit() does: _divide_samples, the CUDA-graph captures of the first epoch, the per-epoch loss read-back."""
    import torch
    from cvae_gan_b200 import CVAEGAN, config, datasets
    from cvae_gan_b200.datasets import TrDataset
    g = torch.Generator().manual_seed(0)
    xs, ys = [], []
    for k in range(K_):
        c = torch.rand(F_, generator=g)
        xs.append((c + 0.08 * torch.randn(rows_per_class, F_, generator=g)).clamp(0, 1))
        ys.append(torch.full((rows_per_class,), k, dtype=torch.long))
    datasets.tr_samples, datasets.tr_labels = torch.cat(xs), torch.cat(ys)
    datasets.feature_num, datasets.label_num = F_, K_
    gc = config.gan_config
    keep = (gc.batch_size, gc.epochs)
    gc.batch_size, gc.epochs = BATCH_PER_GPU, epochs
    try:
        torch.manual_seed(0)
        gan = CVAEGAN()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gan.fit(TrDataset())
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t1 = time.perf_counter()
        gan.fit(TrDataset())            # a second fit: program / kernel images are warm, the graphs are captured again
        torch.cuda.synchronize()
        dt2 = time.perf_counter() - t1
        n_q = 200_000
        # a label this young classifier accepts at all (the reference's loop gives up after 20 empty chunks of 10)
        accs = [float(gan.engine.generate_filter(lab, 20_000, 0.0, seed=5, capacity=1)[2].item()) for lab in range(K_)]
        q_label = int(max(range(K_), key=lambda lab: accs[lab]))
        t2 = time.perf_counter()
        q = gan.generate_qualified_samples(q_label, n_q, 0.0)
        dq = time.perf_counter() - t2
        samples = OPT_STEPS * BATCH_PER_GPU * K_ * epochs
        out = {"value": samples / dt2, "unit": "samples/s", "first_fit_value": samples / dt, "epochs": epochs, "rows": rows_per_class * K_,
               "seconds": dt2, "first_fit_seconds": dt,
               "api": "CVAEGAN().fit(TrDataset()) at batch 4096: _divide_samples + graph capture + epochs x K label visits + loss read-back",
               "generate_qualified_samples": {"requested": n_q, "returned": int(q.shape[0]) if q.dim() == 2 else 0, "seconds": dq,
                                              "rows_per_s": (int(q.shape[0]) if q.dim() == 2 else 0) / dq, "threshold": 0.0,
                                              "label": q_label, "api": "gan.generate_qualified_samples(label, 200000, 0.0) -> CPU tensor"}}
        gan.engine.close()
        return out
    finally:
        gc.batch_size, gc.epochs = keep


# ---------------------------------------------------------------------------------------------------------
# second headline metric (BASELINE.json configs[3]): minority-class generation + classifier-confidence filter
# ---------------------------------------------------------------------------------------------------------
GEN_ROWS_PER_GPU = int(os.environ.get("CVG_BENCH_GEN_ROWS", "12500000"))   # 100 M rows over 8 GPUs
# fused path: 2 * (75 648 + 43 840) FLOP per generated row (SURVEY.md 8d); standalone filter: 4F + 4K + a(4F + 8) B/row
GEN_FLOP_PER_ROW = 2 * (75_648 + 43_840)


K_OTIDS = 4
OTIDS_FRACTIONS = (0.90, 0.06, 0.03, 0.01)
FILTER_TRAIN_EPOCHS = int(os.environ.get("CVG_BENCH_FILTER_EPOCHS", "400"))


def trained_otids_engine(dev, world, rank):
    """CAN-HCRL-OTIDS-shaped model for BASELINE.json configs[3] (SURVEY 8d C4): K = 4 classes with fractions
    [0.90, 0.06, 0.03, 0.01] of 1 M synthetic rows, trained here for FILTER_TRAIN_EPOCHS epochs (label visits of 5 D + 5 C +
    3 E/G steps at batch 4096, lambda_class = 0.25) so that the classifier is a usable filter at the reference's threshold
    of 0.5 (gan_config.py:20).  Rank 0 trains; the other ranks receive its parameters."""
    import torch
    import torch.distributed as dist
    from cvae_gan_b200 import models
    from cvae_gan_b200.engine import Engine
    eng = Engine(F_, K_OTIDS, Z_, max_batch=BATCH_PER_GPU)
    torch.manual_seed(1)
    mods = [models.CVAEGANEncoderModel(F_, K_OTIDS, Z_), models.CVAEGANGeneratorModel(Z_, K_OTIDS, F_),
            models.CVAEGANDiscriminatorModel(F_, K_OTIDS), models.CVAEGANClassifierModel(F_, K_OTIDS)]
    for net, m in enumerate(mods):
        eng.load_state(net, m.state_dict())
    t_train = 0.0
    if rank == 0:
        g = torch.Generator(device="cpu").manual_seed(7)
        tabs = []
        for k, fr in enumerate(OTIDS_FRACTIONS):
            c = torch.rand(F_, generator=g)
            n = int(1_000_000 * fr)
            tabs.append((c.to(dev) + 0.08 * torch.randn(n, F_, device=dev)).clamp_(0, 1).contiguous())
        eng.ctl_set(seed=4321, counter=0, lambda_class=0.25)
        loss = torch.zeros(OPT_STEPS, 4, device=dev)
        graphs = {}
        for label in range(K_OTIDS):
            eng.visit(label, BATCH_PER_GPU, class_rows=tabs[label], loss_out=loss)
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                eng.visit(label, BATCH_PER_GPU, class_rows=tabs[label], loss_out=loss)
            graphs[label] = gr
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for e in range(FILTER_TRAIN_EPOCHS):
            for label in range(K_OTIDS):
                graphs[label].replay()
        torch.cuda.synchronize()
        t_train = time.perf_counter() - t0
        del graphs
    if world > 1:
        for net in range(4):
            dist.broadcast(eng.params[net], src=0)
            dist.broadcast(eng.state[net], src=0)
    return eng, {"epochs": FILTER_TRAIN_EPOCHS, "label_visits": FILTER_TRAIN_EPOCHS * K_OTIDS, "seconds": t_train,
                 "class_fractions": list(OTIDS_FRACTIONS), "rows": 1_000_000, "batch": BATCH_PER_GPU}


def run_filter_leg(eng_unused, dev, world, rank, pk, iters=3):
    """Generated rows/s and accepted rows/s of the one-pass generate -> classify -> threshold -> compact kernel
    (rows sharded by global row index, no collective), plus the standalone filter kernel against the HBM roofline.
    Named configuration: OTIDS-shaped K = 4 model trained in this run, a MINORITY label, threshold 0.5."""
    import torch
    import torch.distributed as dist
    eng, train_info = trained_otids_engine(dev, world, rank)
    K_ = K_OTIDS
    n, thr = GEN_ROWS_PER_GPU, 0.5
    # acceptance of the minority labels at the reference's threshold (100 k rows each, same rows on every rank)
    acc = {}
    for lab in (1, 2, 3):
        _, _, cnt, _, _ = eng.generate_filter(lab, 100_000, thr, seed=99, row_offset=0, capacity=1)
        acc[lab] = float(cnt.item()) / 100_000
    label = max(acc, key=lambda k: acc[k])
    fallback = False
    if acc[label] < 0.01:
        # labelled fallback (not the named configuration): lower the threshold until the classifier accepts something
        fallback = True
        for t in (0.35, 0.25, 0.0):
            for lab in range(K_):
                _, _, cnt, _, _ = eng.generate_filter(lab, 100_000, t, seed=99, row_offset=0, capacity=1)
                if float(cnt.item()) / 100_000 >= 0.01:
                    label, thr = lab, t
                    break
            else:
                continue
            break
    row_offset = rank * n
    x_out = torch.empty(n, F_, device=dev)
    idx_out = torch.empty(n, dtype=torch.int64, device=dev)
    host_x = torch.empty(n, F_).pin_memory()
    from cvae_gan_b200._lib import check
    from cvae_gan_b200.engine import _ptr, _stream

    def gen_filter():
        eng.count_buf.zero_()
        check(eng.lib.cvg_generate_filter(eng.h, label, n, thr, None, 99, row_offset, _ptr(x_out), _ptr(idx_out), n,
                                          _ptr(eng.count_buf), None, None, _stream()))

    def timed(fn, k, warm):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / k

    # the NAMED configuration first: minority label, threshold 0.5 - measured even when the acceptance is ~0
    named = None
    if fallback:
        nl = max(acc, key=lambda k: acc[k])
        keep_lt = (label, thr)
        label, thr = nl, 0.5
        ms_n = timed(gen_filter, iters, 2)
        acc_n = torch.tensor([float(eng.count_buf.item())], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(acc_n)
        named = {"label": nl, "threshold": 0.5, "ms_per_pass": ms_n, "generated_rows_per_s": n * world / (ms_n * 1e-3),
                 "accepted_rows_per_s": float(acc_n.item()) / (ms_n * 1e-3), "acceptance_rate": float(acc_n.item()) / (n * world),
                 "note": "the classifier separates the REAL classes (accuracy 1.0, confidence ~0.99 after the training above) but the "
                         "generator trained by the reference's algorithm at these settings does not carry the class into its samples "
                         "(recon loss flat, KL -> 0; the CPU oracle shows the same curve, tools/diag_longrun.py), so nothing "
                         "passes 0.5: `value` is therefore measured at the lowered threshold and flagged threshold_fallback"}
        label, thr = keep_lt
    ms = timed(gen_filter, iters, 3)
    accepted = int(eng.count_buf.item())
    dbg = None
    if os.environ.get("CVG_TC_DBG") == "1":       # development: per-role cycle split of the fused kernel
        cnt = torch.zeros(32, dtype=torch.int64, device=dev)
        check(eng.lib.cvg_debug_tc_counters(eng.h, _ptr(cnt)))
        gen_filter()
        torch.cuda.synchronize()
        check(eng.lib.cvg_debug_tc_counters(eng.h, None))
        tiles = (n + 127) // 128 if os.environ.get("CVG_TC_MODE", "128") == "128" else (n + 63) // 64
        dbg = {k: v / tiles for k, v in zip(("issuer_wait_act", "issuer_wait_weights", "issuer_wait_stage", "issuer_total",
                                              "epi_wait_acc", "epi_input", "epi_total", "issue", "L0", "L1", "L2", "L3", "L4", "L5", "L6", "L7", "epi_tmem_ld(64) / plane_free wait(128)", "epi_fence", "E0", "E1", "E2", "E3", "E4", "E5", "E6", "E7"), cnt.tolist())}

    def gen_filter_e2e():
        gen_filter()
        c = int(eng.count_buf.item())                      # D2H of the count, host sync
        host_x[:c].copy_(x_out[:c], non_blocking=True)     # accepted rows to pinned host memory
        torch.cuda.current_stream().synchronize()

    ms_e2e = timed(gen_filter_e2e, iters, 1)
    tot = torch.tensor([accepted], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tot)
    accepted_all = float(tot.item())
    gen_rows_s = n * world / (ms * 1e-3)
    out = {
        "metric": "filtered_synth_samples_per_s", "value": accepted_all / (ms * 1e-3), "unit": "accepted rows/s",
        "generated_rows_per_s": gen_rows_s, "acceptance_rate": accepted_all / (n * world), "rows_per_gpu": n,
        "ms_per_pass": ms, "label": label, "threshold": thr, "cycles_per_tile": dbg,
        "config": {"workload": "minority-class generation + classifier-confidence filter, OTIDS shape F=10 K=4 Z=128 "
                               "(BASELINE.json configs[3]): 12.5 M generated rows per GPU, threshold 0.5",
                   "model": train_info, "minority_acceptance_at_thr": {str(k): v for k, v in acc.items()},
                   "threshold_fallback": fallback, "named_config_measured": named},
        "e2e": {"value": accepted_all / (ms_e2e * 1e-3), "generated_rows_per_s": n * world / (ms_e2e * 1e-3),
                "unit": "accepted rows/s", "ms_per_pass": ms_e2e, "d2h_bytes_per_pass": accepted * (F_ * 4) + 8,
                "api": "cvg_generate_filter + count read-back + accepted rows copied to pinned host memory"},
        "roofline_fused": {"bound": "tensor", "kernel": "tc_eval128_kernel (tcgen05 kind::tf32, 3xTF32, 128-row tiles)",
                           "traffic": ncu_traffic().get("tc_eval128_kernel", {}).get("bytes"),
                           "achieved": gen_rows_s / world * GEN_FLOP_PER_ROW / 1e12, "peak": pk["bf16_tflops"],
                           "unit": "TFLOP/s", "frac": gen_rows_s / world * GEN_FLOP_PER_ROW / 1e12 / pk["bf16_tflops"],
                           "note": "algorithmic fp32 FLOP; each costs 3 tf32 MMAs (fp32-accurate split), tf32 peak is half the "
                                   "bf16 peak quoted here: the tensor pipe does 6x the algorithmic FLOP in bf16-peak units"},
    }
    # standalone memory-bound filter over materialised tensors (the kernel judged against the HBM roofline)
    m = min(n, 12_500_000)
    g = torch.Generator(device=dev).manual_seed(5)
    x = torch.rand(m, F_, device=dev, generator=g)
    lg = 3.0 * torch.randn(m, K_, device=dev, generator=g)

    def standalone():
        eng.count_buf.zero_()
        check(eng.lib.cvg_filter_compact(_ptr(x), _ptr(lg), m, F_, K_, label, thr, 0, _ptr(x_out), _ptr(idx_out), m,
                                         _ptr(eng.count_buf), _stream()))

    ms_f = timed(standalone, 10, 3)
    acc_f = int(eng.count_buf.item())
    # bytes the kernel must move: logits of every row, x of ACCEPTED rows only (read + written) and their indices
    byts = m * (4 * K_) + acc_f * (4 * F_ + 4 * F_ + 8)
    byts_survey = m * (4 * F_ + 4 * K_) + acc_f * (4 * F_ + 8)
    out["roofline_filter"] = {"bound": "hbm", "kernel": "filter_compact_stream_kernel", "achieved": byts / (ms_f * 1e-3) / 1e9,
                              "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": byts / (ms_f * 1e-3) / 1e9 / pk["hbm_gbs"],
                              "rows": m, "acceptance_rate": acc_f / m, "bytes_per_row_model": "4K + a(4F + 4F + 8): x of rejected rows is never read",
                              "survey_model_gbs": byts_survey / (ms_f * 1e-3) / 1e9, "survey_model": "4F + 4K + a(4F + 8)",
                              "survey_model_frac": byts_survey / (ms_f * 1e-3) / 1e9 / pk["hbm_gbs"],
                              "rows_per_s": m / (ms_f * 1e-3), "ms": ms_f,
                              "traffic": ncu_traffic().get("filter_compact_stream_kernel", {}).get("bytes")}
    if world == 1:
        eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-filter", action="store_true", help="skip the generation + filter leg")
    ap.add_argument("--no-fit", action="store_true", help="skip the CVAEGAN.fit drop-in leg")
    ap.add_argument("--no-wide", action="store_true", help="skip the widened-model leg (BASELINE.json configs[4], fp32, 1 GPU)")
    ap.add_argument("--only-filter", action="store_true", help="dev aid: run only the generation + filter leg")
    ap.add_argument("--quick", action="store_true", help="profiling aid (ncu): resident loop only, no e2e/cpu legs; NOT a bench number")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the losses of the last timed label visit "
                                                          "and the four networks' state after it to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.quick or args.only_filter):
        ap.error("--dump-outputs writes the outputs of the training visits timed by --impl ours (not --quick / --only-filter)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
