#!/usr/bin/env python
"""Benchmark of the VTP hot path on B200 (contract: see the task brief / DESIGN.md §Measurement).

  python bench.py --gpus N --steps K --warmup W            our arm  (one rank per GPU under torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  reference arm: the CPU restatement of the reference's step
                                                           (oracle/train_step.py) on the box's host cores, rank 0 only

Workload (BASELINE.json configs[1]): VTP-Small f16d64, full 3-loss training step (contrastive + DINO/iBOT + recon incl.
LPIPS), batch 256 per GPU, 256x256 synthetic RGB, 2 global + 8 local(96) crops, K=65536 prototypes, AdamW + EMA teacher.
The step runs as ONE captured CUDA graph by default (--graph off = eager launches).  Prints ONE JSON line.

Both arms time the same workload definition; the reference arm's timed steps are a bounded sample of it (--cpu-batch
source images per step, stated in its line).  `cpu_config1` in our line is BASELINE configs[0] (the reference's own
CPU-runnable case: VTP-Small, batch 4, encode->decode, fp32, no_grad) timed on the CPU oracle.
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

METRIC = "images/sec (256x256 encode+decode+3-loss step)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="small")
    ap.add_argument("--batch", type=int, default=256, help="source images per GPU per step")
    ap.add_argument("--prototypes", type=int, default=65536)
    ap.add_argument("--cpu-batch", type=int, default=4, help="source images per step of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lpips", action="store_true", help="reconstruction loss = L1 only")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="run the step as one captured CUDA graph (auto = on)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])), mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _cpu_threads() -> int:
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # the GPU boxes expose 128 logical CPUs; intra-op threading of these small CPU GEMMs stops scaling (and, under a
    # cgroup CPU quota, collapses) long before that — use at most 32 threads and report the number actually used
    return int(os.environ.get("VTP_CPU_THREADS", min(avail, 32)))


def cpu_baseline(args, steps: int, warmup: int):
    """The reference's step restated on the CPU oracle (towers + restated losses incl. LPIPS + autograd + AdamW + EMA),
    bounded sample: `steps` timed steps of `--cpu-batch` source images each.  Returns (cpu_baseline object, s/step)."""
    import torch

    from oracle.train_step import OracleTrainer
    from vtp_b200.config import preset
    from vtp_b200.model import VTPModel
    from vtp_b200.synthetic import make_batch

    cores = _cpu_threads()
    torch.set_num_threads(cores)
    cfg = preset(args.model)
    m = VTPModel(cfg)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    K = args.prototypes
    g = torch.Generator().manual_seed(0)
    D = cfg.vision_embed_dim
    hsd = {"mlp.0.weight": torch.randn(2048, D, generator=g) * 0.02, "mlp.0.bias": torch.zeros(2048),
           "mlp.2.weight": torch.randn(2048, 2048, generator=g) * 0.02, "mlp.2.bias": torch.zeros(2048),
           "mlp.4.weight": torch.randn(256, 2048, generator=g) * 0.02, "mlp.4.bias": torch.zeros(256),
           "last_layer.weight_g": torch.ones(K, 1), "last_layer.weight_v": torch.randn(K, 256, generator=g) * 0.02}
    dims = dict(vision_depth=cfg.vision_depth, vision_num_heads=cfg.vision_num_heads, text_depth=cfg.text_depth,
                text_num_heads=cfg.text_num_heads, decoder_depth=cfg.decoder_depth, decoder_num_heads=cfg.decoder_num_heads)
    lp = None
    if not args.no_lpips:
        from vtp_b200.lpips import random_weights
        lp = random_weights(0)                      # the same frozen seeded-random VGG16 / lin weights as the GPU arm
    tr = OracleTrainer(sd, hsd, dims, n_local=8, mode="bf16", lpips=lp)
    Bc = args.cpu_batch
    batch = make_batch(Bc, vocab=cfg.text_vocab_size)
    for _ in range(warmup):
        tr.step(batch)
    t0 = time.perf_counter()
    for _ in range(steps):
        tr.step(batch)
    dt = (time.perf_counter() - t0) / steps
    return {"value": Bc / dt, "unit": "images/sec", "cores": cores, "kind": "port", "steps_timed": steps, "warmup": warmup,
            "batch": Bc,
            "sample": f"{steps} timed step(s) (+{warmup} warm-up) of the same 3-loss step ({'with' if lp else 'without'} LPIPS) at batch "
                      f"{Bc} instead of {args.batch} (bf16-autocast emulation, torch CPU, {cores} threads), {dt:.2f} s/step"}, dt


def cpu_config1(reps: int = 3):
    """BASELINE.json configs[0] / SURVEY.md §8(d) "CPU baseline timing": VTP-Small, batch 4, encode -> decode, fp32,
    no_grad, exactly the call pattern of tools/test_reconstruction_hf.py:360-372 — on the CPU oracle (kind "port": the
    reference itself cannot travel to the GPU box; the oracle is pinned to it, tests/test_oracle_golden.py)."""
    import torch

    from oracle import vtp_oracle as vo
    from vtp_b200.config import preset
    from vtp_b200.flops import encode_decode_flops
    from vtp_b200.model import VTPModel

    cores = _cpu_threads()
    torch.set_num_threads(cores)
    cfg = preset("small")
    sd = {k: v.detach().clone() for k, v in VTPModel(cfg).state_dict().items()}
    x = torch.randn(4, 3, 256, 256, generator=torch.Generator().manual_seed(1234))
    ts = []
    with torch.no_grad():
        for i in range(reps + 1):
            t0 = time.perf_counter()
            lat = vo.reconstruction_latents(x, sd, depth=cfg.vision_depth, heads=cfg.vision_num_heads)
            vo.decode_latents(lat, sd, depth=cfg.decoder_depth, heads=cfg.decoder_num_heads)
            if i:
                ts.append(time.perf_counter() - t0)
    ts.sort()
    med = ts[len(ts) // 2]
    return {"workload": "VTP-Small f16d64, batch=4 256x256, encode->decode reconstruction only, fp32, no_grad, CPU",
            "value": 4 / med, "unit": "images/sec", "ms_per_call": med * 1e3, "cores": cores, "kind": "port", "reps": reps,
            "gflop_per_image": encode_decode_flops(cfg) / 1e9}


DUMP_SAMPLE = 1 << 21       # elements per sampled array: 2 x 8 MiB of float32


def _canonical_sample(store, names, k: int, seed: int = 0):
    """Indices into the flat buffers of `store` of k elements drawn with a fixed seed from the parameters `names`,
    flattened one after the other in sorted-name order: the sample picks the same parameter elements whatever order and
    alignment the store lays them out in."""
    import torch

    names = sorted(names)
    sizes = torch.tensor([store.f32(n).numel() for n in names])
    offsets = torch.tensor([store.offset[n] for n in names])
    ends = sizes.cumsum(0)
    pos = torch.randint(int(ends[-1]), (k,), generator=torch.Generator().manual_seed(seed)).sort().values
    which = torch.searchsorted(ends, pos, right=True)
    return (offsets[which] + pos - (ends[which] - sizes[which])).to(store.p.device)


def dump_outputs(out_dir: str, tr, loss):
    """What a caller of the training step receives from the last timed step, as float32 .npy files: `loss` (the loss
    vector the step returns) and seeded samples (DUMP_SAMPLE elements each, see _canonical_sample) of the updated student
    parameters (`params`) and of the updated EMA teacher (`teacher`)."""
    import numpy as np

    st = tr.store
    os.makedirs(out_dir, exist_ok=True)
    idx = _canonical_sample(st, st.offset, DUMP_SAMPLE)
    tidx = _canonical_sample(st, [name for name, _, _, teacher in st.specs if teacher], DUMP_SAMPLE)
    arrays = {"loss": loss, "params": st.p[idx], "teacher": st.tp[tidx]}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def workload_config(args, world: int, flops_per_image: float, image_groups=None) -> dict:
    """The `config` object of the JSON line — identical for both arms (the reference arm adds its bounded sample)."""
    B = args.batch
    cfg = {"workload": f"VTP-{args.model} f16d64 full 3-loss training step (contrastive+SSL+recon), batch={B}/GPU",
           "model": "VTP-Small 384/12/6 x3 towers (ASSUMED, SURVEY.md §8d)" if args.model == "small" else args.model,
           "global_batch": B * world, "image": 256, "crops": "2 global 256 + 8 local 96 per image",
           "prototypes": args.prototypes,
           "losses": ["clip", "dino_local", "dino_global", "ibot", "rec_l1"] + ([] if args.no_lpips else ["rec_lpips"]),
           "lpips": (not args.no_lpips) and "VGG16 (frozen, seeded-random weights: pretrained ones need network), weight 1.0",
           "optimizer": "fused AdamW + EMA teacher, in the timed region",
           "l2": "inputs (>1 GB/step) and activations far exceed the 126 MB L2; no reuse across steps",
           "parallelism": f"dp{world}", "flops_per_image": flops_per_image}
    if image_groups is not None:
        cfg["image_groups"] = image_groups
    return cfg


def log(msg):
    if os.environ.get("RANK", "0") == "0":
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        if rank != 0:
            return
        # bounded: at most 2 timed steps (+1 warm-up) of --cpu-batch images — about 10-30 s of CPU work
        n_steps, n_warm = max(1, min(args.steps, 2)), min(args.warmup, 1)
        cb, dt = cpu_baseline(args, steps=n_steps, warmup=n_warm)
        from vtp_b200.config import preset
        from vtp_b200.flops import train_step_flops_per_image
        fl = train_step_flops_per_image(preset(args.model), K=args.prototypes, lpips=not args.no_lpips)
        conf = workload_config(args, args.gpus, fl["total"])
        conf["sample"] = (f"CPU restatement of the reference's step (oracle port, torch CPU, {cb['cores']} threads): each timed "
                          f"step is a bounded sample of {args.cpu_batch} source images of this workload (same crops, prototypes, "
                          f"losses incl. LPIPS, optimiser); {n_steps} step(s) timed after {n_warm} warm-up, whatever --steps/--warmup ask")
        out = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "images/sec", "n_gpus": args.gpus,
               "steps": n_steps, "warmup": n_warm, "steps_requested": args.steps, "warmup_requested": args.warmup,
               "ms_per_step": dt * 1e3, "ms_per_step_is_for_batch": args.cpu_batch, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
               "config": conf,
               "cpu_baseline": cb,
               "e2e": {"value": cb["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(out), flush=True)
        return

    import torch
    import torch.distributed as dist

    from vtp_b200 import lib
    from vtp_b200.config import preset
    from vtp_b200.flops import train_step_flops_per_image
    from vtp_b200.synthetic import BatchPrefetcher, batch_bytes, make_batch, to_device
    from vtp_b200.train import TrainConfig, VTPTrainer

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = preset(args.model)
    # VTP-Base/Large at 256 images per GPU: size the SSL / reconstruction image groups for the 180 GB of HBM
    # (vtp_b200/memory.py; (0, 0) = whole batch in one pass, which is what VTP-Small uses)
    from vtp_b200.memory import suggest_chunks
    ssl_chunk, rec_chunk = suggest_chunks(cfg, args.batch, head_out_dim=args.prototypes, lpips=not args.no_lpips)
    tc = TrainConfig(head_out_dim=args.prototypes, ssl_chunk=ssl_chunk, rec_chunk=rec_chunk)
    tr = VTPTrainer(cfg, tc, device=dev)
    if not args.no_lpips:
        tr.enable_lpips(seed=0, chunk=int(os.environ.get("VTP_LPIPS_CHUNK", "32")))
    log(f"trainer built: {tr.store.n / 1e6:.1f}M params")
    B = args.batch
    host = make_batch(B, vocab=cfg.text_vocab_size, seed=1234 + rank, pin=True)
    resident = to_device(host, dev, non_blocking=False)
    log(f"batch ready: {batch_bytes(host) / 2**20:.0f} MiB/step")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    use_graph = args.graph != "off"
    step_fn = tr.train_step
    if use_graph:
        # warm-up steps run inside capture_step (they are real, eager steps), then one step is captured without executing
        tr.capture_step(resident, warmup=max(args.warmup, 1))
        torch.cuda.synchronize()
        log(f"step captured: {tr.graph_launches} kernels per replay, peak mem {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")
        step_fn = tr.replay_step
        tr.replay_step()           # one replay before timing (graph upload)
        torch.cuda.synchronize()
    else:
        for i in range(args.warmup):
            tr.train_step(resident)
            torch.cuda.synchronize()
            log(f"warmup {i} done, peak mem {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- device-resident timing ("value"): inputs already in HBM (the graph's static buffers / the resident batch)
    l0 = lib.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        loss = tr.replay_step() if use_graph else tr.train_step(resident)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = lib.LAUNCHES - l0
    log(f"device-resident: {ms / args.steps:.1f} ms/step")
    # ---- end-to-end timing: pinned host inputs -> H2D -> step -> D2H of the loss vector, every step
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h2d = batch_bytes(host)
    e2.record()
    pf = BatchPrefetcher(dev)
    pf.put(host)                      # step 0's inputs: exposed
    loss_pin = [torch.empty(8, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_evt = [None, None]
    for i in range(args.steps):
        dev_batch, slot = pf.get()
        if i + 1 < args.steps:
            pf.put(host)              # the next step's 1 GB H2D copy runs on the side stream under this step
        loss = step_fn(dev_batch)     # graph: device-to-device copy into the static inputs (0.3 ms), then one replay
        pf.release(slot)
        loss_pin[i & 1].copy_(loss, non_blocking=True)   # D2H of this step's result, every step ...
        loss_evt[i & 1] = torch.cuda.Event()
        loss_evt[i & 1].record()
        if i >= 1:                    # ... read by the host once the NEXT step is enqueued (what an async logger does):
            loss_evt[(i - 1) & 1].synchronize()          # the launch of step i hides behind step i-1 instead of idling the GPU
            loss_host = loss_pin[(i - 1) & 1].clone()
    loss_evt[(args.steps - 1) & 1].synchronize()
    loss_host = loss_pin[(args.steps - 1) & 1].clone()
    e3.record()
    barrier()
    ms_e2e = max_over_ranks(e2.elapsed_time(e3))
    log(f"end-to-end: {ms_e2e / args.steps:.1f} ms/step")
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tr, loss_host)
        log(f"outputs of the last step written to {args.dump_outputs}")
    # ---- dominant kernel: the tcgen05 GEMM (gemm_kernel<256,4,NONE>), timed live on its largest recurring shape on the
    #      hot path: the FFN fc1 projection of the SSL student pass (bias, bf16 out; the SwiGLU gate is a separate pass)
    Mg, Ng, Kg = 2 * B * 257, 2 * tr.hs, tr.D
    A = torch.randn(Mg, Kg, device=dev).to(torch.bfloat16)
    Wt = torch.randn(Ng, Kg, device=dev).to(torch.bfloat16)
    bias = torch.zeros(Ng, device=dev)
    outg = torch.empty(Mg, Ng, device=dev, dtype=torch.bfloat16)
    for _ in range(3):
        lib.gemm(A, Wt, outg, M=Mg, N=Ng, K=Kg, bias=bias)
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    torch.cuda.synchronize()
    g0.record()
    for _ in range(reps):
        lib.gemm(A, Wt, outg, M=Mg, N=Ng, K=Kg, bias=bias)
    g1.record()
    torch.cuda.synchronize()
    gemm_ms = g0.elapsed_time(g1) / reps
    gemm_tflops = 2.0 * Mg * Ng * Kg / (gemm_ms * 1e-3) / 1e12
    traffic, traffic_src = None, None
    try:  # DRAM bytes of this very launch (same M, N, K) from the committed ncu --set full capture under profiles/ — ncu
        # cannot run inside the timed bench, so the number is stamped with the capture it came from
        with open(os.path.join(ROOT, "profiles", "gemm_fc1_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("M") == Mg and tj.get("N") == Ng and tj.get("K") == Kg:
            traffic, traffic_src = tj["dram_bytes"], tj.get("source", "profiles/gemm_fc1_traffic.json")
    except Exception:
        pass

    def shutdown():
        """Release the step graph BEFORE the NCCL communicator (NCCL cannot destroy a communicator whose collectives live in a
        CUDA graph: the first 2-GPU graph run of round 2 hung right here), with a hard-exit watchdog behind it — the JSON
        line is already flushed at that point."""
        if world > 1:
            t = threading.Timer(30.0, lambda: os._exit(0))
            t.daemon = True
            t.start()
            tr.release_graph()
            dist.destroy_process_group()
            t.cancel()

    if rank != 0:
        shutdown()
        return
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak_burst = peaks.get("bf16_tflops", 1590.0)
    peak_sust = peaks.get("bf16_tflops_sustained", 1400.0)
    src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    fl = train_step_flops_per_image(cfg, K=args.prototypes, lpips=not args.no_lpips)
    imgs = B * world * args.steps
    value = imgs / (ms * 1e-3)
    step_tflops = fl["total"] * B / (ms / args.steps * 1e-3) / 1e12  # per GPU
    out = {
        "metric": METRIC, "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args, world, fl["total"], {"ssl_chunk": ssl_chunk, "rec_chunk": rec_chunk}),
        "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "images/sec", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": int(loss_host.numel() * 4), "ms_per_step": ms_e2e / args.steps,
                "pipeline": "vtp_b200.synthetic.BatchPrefetcher: pinned host batch of step i+1 copied on a side stream "
                            "(2 device buffers) while step i runs; step 0's copy exposed; every step's loss vector is copied D2H right after the "
                            "step and read by the host one step later (after step i+1 is enqueued), the last one before the clock stops"},
        "gpu_launches": launches,
        "launch_mode": (f"one CUDA graph replay per step ({tr.graph_launches} kernels of libvtp_b200.so inside)" if use_graph
                        else "eager: one host launch per kernel"),
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": f"vtp::gemm_kernel<256,4,NONE,cluster2,TMA-store epilogue> FFN fc1 GEMM M={Mg} N={Ng} K={Kg} (+bias, bf16 out), "
                               f"timed ISOLATED on synthetic operands after the step loop ({reps} launches, CUDA events)",
                     "achieved": gemm_tflops, "peak": peak_burst, "unit": "TFLOP/s", "frac": gemm_tflops / peak_burst,
                     "peak_source": src + " burst (kernel timed alone)", "traffic": traffic, "traffic_source": traffic_src,
                     "algorithmic_flops_per_launch": 2.0 * Mg * Ng * Kg,
                     "algorithmic_bytes_per_launch": 2.0 * (Mg * Kg + Ng * Kg + Mg * Ng),
                     "step": {"achieved": step_tflops, "peak": peak_sust, "frac": step_tflops / peak_sust,
                              "note": "whole-step algorithmic FLOPs (vtp_b200/flops.py) / step time vs sustained bf16 peak"}},
        "loss": [round(float(x), 5) for x in loss_host[:6]],
    }
    if world == 1 and not args.no_cpu_baseline:
        log("cpu baseline ...")
        cb, _ = cpu_baseline(args, steps=2, warmup=1)   # ~20 s of CPU work on the box's 32 threads
        out["cpu_baseline"] = cb
        out["cpu_config1"] = cpu_config1()              # BASELINE configs[0]: the reference's own CPU-runnable case
    extra = os.path.join(ROOT, "profiles", "extra_configs_r2.json")
    if os.path.exists(extra):                           # BASELINE configs[2..4]: committed hardware runs of this round
        try:
            with open(extra) as f:
                out["extra_configs"] = json.load(f)
        except Exception:
            pass
    print(json.dumps(out), flush=True)
    shutdown()


if __name__ == "__main__":
    main()
