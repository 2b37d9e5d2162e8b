#!/usr/bin/env python
"""bench.py — BASELINE.json metric: text-line-crops/sec (recognition), config 2.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE config 2 / SURVEY.md §8d): B = 256 synthetic 48x512 uint8 line crops per GPU -> 56x560,
160 patches, 46-token prompt each; declared synthetic model SYN-REC (vision tower = reference defaults,
decoder 12 x 1280, GQA 16/4, vocab 65 792), bf16, greedy decode max_tokens = 128 with early exit disabled
(all 256 rows run 1 prefill + 127 decode steps).  A "step" is one pass of that hot path over one 256-crop batch.

  value : crops/s, whole job, inputs (fp32 tiles + index plan) already resident in HBM when the clock starts
  e2e   : crops/s through the public API (RecognitionRunner.run_preprocessed) from pinned HOST buffers,
          host->device copies of tiles/plan and device->host reads of tokens/scores/boxes inside the timed region
  roofline     : dominant kernel = the tcgen05 GEMM in the HBM-bound decode step (see DESIGN.md §5)
  cpu_baseline : oracle port (fp32 PyTorch restatement of the reference modules) on this box's host cores,
                 bounded sample, rank 0 only

Secondary objects in the same JSON line (never in the headline region; a failure is reported inside the object): `detection`
(config 3), `layout` / `table_rec` (config 4), `ocr_pipeline` (config 5, with device and with host crop preprocessing),
`e2e_from_crops` (recognition from uint8 crops with SuryaOCRProcessor's resizes / normalisation / tiling inside the timed region:
sb_rec_preprocess on the device vs the OpenCV thread pool; N = 1 only), `ocr_error` (DistilBERT classifier; N = 1 only),
`gpu_eager_baseline` (the reference algorithm in PyTorch eager on the same GPU).

Multi-GPU (torchrun, one rank per GPU): replicas over independent crop batches (weak scaling); one NCCL
broadcast of the packed weights at init, one all_gather of the result tensors per step.
`--impl reference` times the reference algorithm's CPU path (the oracle port: the reference is Python, so there is nothing
to compile) on all host threads, same metric/config.
`--dump-outputs DIR` writes what the timed path returned in its last step (rank 0's replica) as DIR/{tokens,scores,bboxes}.npy;
the inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "text-line-crops/sec (recognition)"
B_PER_GPU = 256
MAX_TOKENS = 128
CROP_H, CROP_W = 48, 512


_T0 = time.time()


def log(msg):
    print(f"[bench +{time.time() - _T0:6.1f}s] {msg}", file=sys.stderr, flush=True)


def host_threads() -> int:
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, min(n, 64))


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
CPU_CROPS, CPU_STEPS = 32, 33   # bounded sample: the reference's CPU batch (surya/recognition/__init__.py:81), prefill + 32 decode steps


def host_info():
    """What the CPU arm ran on: round 1 saw 0.71 vs 3.49 crops/s on two boxes with the same thread count."""
    model = "?"
    try:
        for line in open("/proc/cpuinfo"):
            if line.lower().startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    try:
        load = os.getloadavg()[0]
    except OSError:
        load = None
    return {"cpu_model": model, "logical_cpus": os.cpu_count(), "affinity": aff, "loadavg_1m": load,
            "torch_threads": torch.get_num_threads(), "torch_interop_threads": torch.get_num_interop_threads()}


def cpu_oracle_sample(n_crops: int, steps: int, threads: int):
    """Oracle port of the reference CPU path (fp32, all modules of the path): prefill + (steps-1) decode steps over
    n_crops crops.  Returns a callable giving (seconds for prefill+steps, seconds extrapolated to MAX_TOKENS)."""
    from oracle import rec_oracle as O
    from surya_b200.config import syn_rec
    from surya_b200.synth import rec_state_dict, rec_synthetic_crops

    torch.set_num_threads(threads)
    cfg = syn_rec()
    sd = rec_state_dict(cfg, seed=0)
    crops = list(rec_synthetic_crops(n_crops, CROP_H, CROP_W, seed=1234))
    batch = O.build_batch(crops, cfg)

    def one():
        t0 = time.perf_counter()
        O.greedy_decode(sd, cfg, batch, 1, torch.float32)            # prefill only
        t_pre = time.perf_counter() - t0
        t0 = time.perf_counter()
        O.greedy_decode(sd, cfg, batch, steps, torch.float32)        # prefill + (steps - 1) decode steps
        t_all = time.perf_counter() - t0
        per_step = max(t_all - t_pre, 0.0) / max(1, steps - 1)
        return t_all, t_pre + per_step * (MAX_TOKENS - 1)

    return one


def cpu_sample_text(n_crops, steps):
    return (f"{n_crops} crops (the reference's CPU batch size): prefill + {steps - 1} decode steps executed (fp32 oracle port of the "
            f"reference modules); crops/s = crops / (t_prefill + t_decode_step x {MAX_TOKENS - 1}), decode extrapolated to {MAX_TOKENS} tokens")


def cpu_baseline_run(repeats: int):
    threads = host_threads()
    one = cpu_oracle_sample(CPU_CROPS, CPU_STEPS, threads)
    runs = []
    for i in range(repeats):
        t_run, t_full = one()
        log(f"cpu arm run {i}: executed {t_run:.1f}s, full-length estimate {t_full:.1f}s")
        runs.append(t_full)
    best = min(runs)
    return {"value": CPU_CROPS / best, "unit": "crops/s", "cores": threads, "kind": "port",
            "sample": cpu_sample_text(CPU_CROPS, CPU_STEPS) + f"; best of {repeats} (all: {[round(CPU_CROPS / r, 3) for r in runs]} crops/s)",
            "host": host_info()}, best


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    log(f"reference arm: {host_threads()} threads")
    cpu, best = cpu_baseline_run(3 if args.steps >= 3 else max(1, args.steps))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "crops/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": 0, "ms_per_step": best * 1e3 * B_PER_GPU / CPU_CROPS, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": _config(args.gpus),
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "crops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ PyTorch-eager GPU arm
def gpu_eager_baseline(dev, steps_rec=MAX_TOKENS):
    """The bar the kernels have to beat (SURVEY.md §8d, VERDICT r1 #6): the reference ALGORITHM in plain PyTorch eager on the
    same B200 — cuBLAS GEMMs, F.scaled_dot_product_attention, DynamicCache-style concatenated KV (oracle/rec_oracle.py with
    FAST_ATTENTION, oracle/det_oracle.py), bf16 recognition / fp16 detection, same synthetic weights, same inputs, same work
    (256 crops x 128 tokens; 32 pages).  Secondary object, not the driver's reference arm."""
    from oracle import det_oracle as D
    from oracle import rec_oracle as O
    from surya_b200.config import det_default, syn_rec
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages, rec_state_dict, rec_synthetic_crops

    out = {}
    cfg = syn_rec()
    dt = torch.bfloat16
    sd = {k: v.to(dev, dt) for k, v in rec_state_dict(cfg, seed=0).items()}
    crops = list(rec_synthetic_crops(B_PER_GPU, CROP_H, CROP_W, seed=1234))
    b = O.build_batch(crops, cfg)
    batch = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in b.items()}
    O.FAST_ATTENTION = True
    try:
        def run():
            return O.greedy_decode(sd, cfg, batch, steps_rec, dt)
        run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tok = run()[0]
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        out["recognition"] = {"value": B_PER_GPU / (ms * 1e-3), "unit": "crops/s", "ms_per_step": ms, "dtype": "bf16",
                              "what": "oracle/rec_oracle.py on cuda: cuBLAS + SDPA (flash / mem-efficient), torch.cat KV cache, "
                                      "one host-free greedy loop of 1 prefill + 127 decode steps",
                              "distinct_tokens_row0": len(set(tok[0].tolist()))}
    finally:
        O.FAST_ATTENTION = False
    del sd, batch
    torch.cuda.empty_cache()
    dcfg = det_default()
    dsd = {k: v.to(dev, torch.float16) for k, v in det_state_dict(dcfg, 0).items()}
    x = det_normalize(det_synthetic_pages(32, 1024, seed=1234)).to(dev, torch.float16)

    def det():
        outs = [D.forward(dsd, dcfg, x[i:i + 8]) for i in range(0, 32, 8)]      # 8-page chunks bound the eager path's workspace
        return torch.cat(outs, 0)
    det()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        det()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    out["detection"] = {"value": 32 / (ms * 1e-3), "unit": "pages/s", "ms_per_step": ms, "dtype": "f16",
                        "what": "oracle/det_oracle.py on cuda: cuDNN convolutions (NCHW, eager), BatchNorm not folded"}
    return out


def dump_outputs(out_dir, prefill: dict, hist: dict) -> None:
    """Tokens / scores / boxes of one resident step laid out as RecognitionRunner.run_preprocessed returns them ([crops, MAX_TOKENS]
    and [crops, MAX_TOKENS, 6], the prefill's token first): integers as float64 (exact), scores as float32.  1.9 MB at B = 256."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    arrays = {"tokens": torch.cat([prefill["tok"][None], hist["tok"]], 0).T.double(),
              "scores": torch.cat([prefill["score"][None], hist["score"]], 0).T.float(),
              "bboxes": torch.cat([prefill["bbox"][None], hist["bbox"]], 0).transpose(0, 1).double()}
    for name, t in arrays.items():
        np.save(d / f"{name}.npy", t.contiguous().cpu().numpy())
    log(f"outputs of the last timed step written to {d}")


def _config(n_gpus):
    return {"workload": f"recognition: {B_PER_GPU} synthetic {CROP_H}x{CROP_W} line crops per GPU, greedy decode "
                        f"max_tokens={MAX_TOKENS} (1 prefill + {MAX_TOKENS - 1} decode steps, early exit off), SYN-REC",
            "model": "SYN-REC (declared synthetic: enc 8x1280/16h/I3420, dec 12x1280 GQA16/4 I3420, vocab 65792)",
            "global_batch": B_PER_GPU * n_gpus, "crops_per_gpu": B_PER_GPU, "max_tokens": MAX_TOKENS,
            "parallelism": f"replicas x{n_gpus} (independent crop batches)",
            "l2": "no flush: per-step working set (0.96 GB weights + 0.5 GB KV + 1.2 GB activations) >> 126 MB L2"}


# ------------------------------------------------------------------------------------------------ GPU arm
def decode_gemm_roofline(eng, peaks, reps=20):
    """Live CUDA-event timing of the GEMM launches of ONE decode step (B=256), replayed as a CUDA graph over the
    engine's real weight tensors.  achieved = algorithmic bytes per launch / average launch duration."""
    from surya_b200 import ops
    from surya_b200.config import align

    cfg = eng.cfg
    d = cfg.decoder
    dev, dt = eng.device, eng.dtype
    B, D = B_PER_GPU, d.hidden_size
    Q = (d.num_attention_heads + 2 * d.num_key_value_heads) * d.head_dim
    Ip = align(d.intermediate_size, 8)
    base = 15 + 10 * cfg.vision_encoder.depth
    x = torch.randn(B, D, device=dev).to(dt)
    ao = torch.randn(B, d.num_attention_heads * d.head_dim, device=dev).to(dt)
    qkv = torch.empty(B, Q, device=dev, dtype=dt)
    act = torch.empty(B, Ip, device=dev, dtype=dt)
    logits = torch.empty(B, cfg.vocab_size, device=dev, dtype=dt)
    calls, nbytes, flops = [], 0, 0

    def add(a, w, out, **kw):
        nonlocal nbytes, flops
        calls.append((a, w, out, kw))
        nbytes += (a.numel() + w.numel() + out.numel()) * 2 + (out.numel() * 2 if kw.get("residual") is not None else 0)
        flops += 2 * a.shape[0] * w.shape[0] * w.shape[1]

    for l in range(d.num_hidden_layers):
        w = eng.weights[base + 5 * l: base + 5 * (l + 1)]
        add(x, w[0], qkv, bias=w[1], rms_eps=d.rms_norm_eps)                   # RMSNorm folded: 1/rms computed inside the GEMM
        add(ao, w[2], x, residual=x)
        add(x, w[3], act, act="silu", swiglu=True, rms_eps=d.rms_norm_eps)
        add(act, w[4], x, residual=x, splitk=True)      # the engine's decode step lets the down projection use split-K
    add(x, eng.weights[7], logits, bias=eng.weights[9], rms_eps=d.rms_norm_eps, argmax_only=True)

    def run():
        for a, w, out, kw in calls:
            ops.gemm(a, w, out=out, **kw)

    run()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        run()
        with torch.cuda.graph(g, stream=s):
            run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g.replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / reps
    n = len(calls)
    achieved = nbytes / n / (ms_step / n * 1e-3) / 1e9
    traffic = None          # DRAM bytes per launch from the committed ncu capture of the same launches (profiles/)
    tp = Path(__file__).resolve().parent / "profiles" / "decode_gemm_traffic.json"
    if tp.exists():
        traffic = json.loads(tp.read_text()).get("dram_bytes_per_launch")
    return {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
            "traffic": traffic, "traffic_src": "profiles/decode_gemm_traffic.json (ncu dram__bytes_read+write, per launch)",
            "kernel": "gemm_tn_kernel / gemm_splitk_kernel (tcgen05), decode-step launches", "launches_per_decode_step": n,
            "alg_bytes_per_launch": nbytes / n, "avg_launch_us": ms_step / n * 1e3, "gemm_ms_per_decode_step": ms_step,
            "gemm_tflops_in_decode": flops / (ms_step * 1e-3) / 1e12, "peak_src": peaks["src"]}, ms_step


def detection_bench(dev, peaks, world, steps, warmup):
    """BASELINE config 3 (secondary metric pages/sec): 32 synthetic 1024x1024 pages per GPU, EfficientViT-L seg
    forward (default config, fp16, BN folded) + x4 bilinear upsample to fp32 on the device."""
    import torch.distributed as dist

    from surya_b200.config import det_default
    from surya_b200.detection import DetEngine, detect_pages_host, detect_text_front_host
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages

    B, S = 32, 1024
    cfg = det_default()
    eng = DetEngine(cfg, det_state_dict(cfg, 0), torch.float16, device=dev, max_batch=B, max_hw=(S, S))
    pages_u8 = det_synthetic_pages(B, S, seed=1234)                       # uint8 [B, S, S, 3]: what the reference's processor receives
    u8_host = (pages_u8 if torch.is_tensor(pages_u8) else torch.from_numpy(pages_u8)).contiguous().pin_memory()
    x_host = det_normalize(pages_u8).half().pin_memory()
    x = x_host.to(dev)
    out_host = torch.empty((B, 2, S, S), dtype=torch.float32).pin_memory()

    def timed(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    def resident():
        eng.forward(x)

    def e2e():
        detect_pages_host(eng, x_host, out_host, chunk=8)
        torch.cuda.synchronize()

    def e2e_front():      # post-processing front half on the device: 16-bit text map + mask + thresholds come back
        detect_text_front_host(eng, u8_host, chunk=16)
        torch.cuda.synchronize()

    for _ in range(max(3, warmup)):
        resident()
    ms = timed(resident, steps) / steps
    e2e()
    ms_e2e = timed(e2e, max(1, min(steps, 3))) / max(1, min(steps, 3))
    e2e_front()
    ms_front = timed(e2e_front, max(1, min(steps, 3))) / max(1, min(steps, 3))
    # strong scaling (BASELINE config 3 / SURVEY.md §8d): the SAME 32 pages split 32/G over the ranks through the product's
    # sharding helper, heat maps all-gathered over NCCL in page order
    strong = None
    if world > 1:
        from surya_b200 import shard

        meta = ((cfg.num_labels, S // 4, S // 4), torch.float16)

        def strong_step():
            return shard.sharded_pages(lambda lo, hi: eng.forward(x[lo:hi]), B, device=dev, result_meta=meta)

        for _ in range(3):
            strong_step()
        ms_s = timed(strong_step, steps) / steps
        strong = {"value": B / (ms_s * 1e-3), "unit": "pages/s", "ms_per_step": ms_s, "pages_total": B, "pages_per_gpu": B / world,
                  "scaling": "strong", "api": "surya_b200.shard.sharded_pages (NCCL all_gather of [pages/G, 2, 256, 256] fp16)"}
    gflop_page = 252.5
    tf = gflop_page * B / (ms * 1e-3) / 1e3
    res = {"metric": "pages/sec (detection)", "value": B * world / (ms * 1e-3), "unit": "pages/s", "ms_per_step": ms,
           "e2e": {"value": B * world / (ms_e2e * 1e-3), "unit": "pages/s", "h2d_bytes_per_step": x_host.numel() * 2,
                   "d2h_bytes_per_step": out_host.numel() * 4,
                   "api": "surya_b200.detection.detect_pages_host (pinned fp16 NCHW pages -> fp32 full-res heatmaps on host; chunks of 8 pipelined over 3 streams)"},
           "e2e_front": {"value": B * world / (ms_front * 1e-3), "unit": "pages/s", "h2d_bytes_per_step": u8_host.numel(),
                         "d2h_bytes_per_step": B * S * S * 3 + B * 16,
                         "api": "surya_b200.detection.detect_text_front_host (pinned uint8 pages, normalised on the device -> fp16 text map "
                                "+ uint8 mask + dynamic thresholds per page; upsample / top-10% mean / binarisation on the device; chunks "
                                "of 16 pipelined over 3 streams — tools/bench_det_e2e.py: smaller chunks lose more in the forward than the overlap wins)"},
           "config": {"workload": f"detection: {B} synthetic {S}x{S} pages per GPU, EfficientViT-L seg forward (default config)",
                      "dtype": "f16"},
           "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                        "frac": tf / peaks["tf_sustained"], "alg_gflop_per_page": gflop_page, "scope": "whole forward"},
           "engine_workspace_gb": eng.workspace_bytes / 1e9, "strong_scaling": strong}
    eng.close()
    return res


def pipeline_bench(dev, world, rank, rec_eng):
    """BASELINE config 5 (secondary): the ocr_text data flow end to end — 64 synthetic 1024x1024 pages per GPU (8 GPUs = the 512
    pages of the config), detect -> host boxes -> polygon crops -> width-sorted recognition (surya_b200.pipeline.OcrPipeline),
    sharded by pages with an all-gather of the per-line results (sharded_ocr).  Pages are white with black text-like bars; with
    synthetic weights the detector fires on a few large regions per page, so this measures the plumbing and the host/device
    split, not a realistic line count."""
    import torch.distributed as dist

    from surya_b200.config import det_default
    from surya_b200.detection import DetEngine
    from surya_b200.pipeline import OcrPipeline, sharded_ocr
    from surya_b200.synth import det_state_dict, det_synthetic_pages

    from surya_b200.recognition import RecEngine

    P, S = 64, 1024
    cfg = det_default()
    det = DetEngine(cfg, det_state_dict(cfg, 0), torch.float16, device=dev, max_batch=8, max_hw=(S, S))
    # detected regions are far larger than the 48x512 benchmark crops (up to ~370 image tokens each): a second engine over the
    # same packed weights with room for long prompts (s_max = prompt + max_tokens) and ragged prefills
    rec = RecEngine(rec_eng.cfg, None, dtype=rec_eng.dtype, device=dev, max_slots=B_PER_GPU + 1, s_max=640, max_patches=65536,
                    max_tokens=32768, packed_weights=rec_eng.weights)
    pages_all = np.concatenate([det_synthetic_pages(P, S, seed=1234 + r, text_like=True) for r in range(world)], 0)

    def run(preprocess):
        pipe = OcrPipeline(det, rec, rec_batch=B_PER_GPU, max_tokens=MAX_TOKENS, det_chunk=8, workers=min(16, host_threads()),
                           preprocess=preprocess)
        sharded_ocr(pipe, pages_all[: 8 * world], MAX_TOKENS, device=dev)          # warm-up (allocations, graph capture)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res, timings = sharded_ocr(pipe, pages_all, MAX_TOKENS, device=dev)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = tt.item()
        return dt, sum(len(p) for p in res), timings

    # the flow with the reference's OpenCV crop preprocessing on the host, then with SURVEY §8 f2's device path (uint8 crops up;
    # pages are not converted to float32 on the host at all) — the second one is the headline of this object
    dt_host, n_lines_host, timings_host = run("host")
    dt, n_lines, timings = run("device")
    det.close()
    rec.close()
    return {"metric": "pages/sec (ocr_text pipeline, end to end)", "value": P * world / dt, "unit": "pages/s", "seconds": dt,
            "pages_total": P * world, "pages_per_gpu": P, "lines_total": n_lines, "lines_per_second": n_lines / dt,
            "preprocess": "device (OcrPipeline(preprocess='device'): sb_rec_preprocess)",
            "breakdown_rank0_s": {k: round(v, 4) for k, v in timings.items()},
            "host_preprocess": {"value": P * world / dt_host, "unit": "pages/s", "seconds": dt_host, "lines_total": n_lines_host,
                                "breakdown_rank0_s": {k: round(v, 4) for k, v in timings_host.items()}},
            "api": "surya_b200.pipeline.sharded_ocr(OcrPipeline) — uint8 pages on the host in, per-line polygons / tokens / scores out",
            "timing": "wall clock around the public call (host post-processing is part of the flow), max over ranks"}


def layout_bench(dev, peaks, world, kind, steps, warmup):
    """BASELINE config 4 (parity-test configs, reported for completeness): 16 synthetic 768x768 pages per GPU through the Swin
    encoder + ADETR decoder; layout = 100 greedy box steps, table_rec = 3-token query prompt + 150 steps (row/column pass)."""
    import torch.distributed as dist

    from surya_b200.config import layout_default, table_default
    from surya_b200.layout import LayoutEngine, layout_greedy, table_greedy
    from surya_b200.synth import (adetr_layout_state_dict, adetr_table_state_dict, layout_synthetic_pages, swin_state_dict,
                                  table_query_tokens)

    B = 16
    cfg = layout_default() if kind == "layout" else table_default()
    sdd = adetr_layout_state_dict(cfg.decoder, 0) if kind == "layout" else adetr_table_state_dict(cfg.decoder, 0)
    eng = LayoutEngine(cfg, swin_state_dict(cfg.encoder, 0), sdd, dtype=torch.float16, device=dev)
    x_host = layout_synthetic_pages(B, cfg.encoder.image_size, seed=1234).half().pin_memory()
    x = x_host.to(dev)
    n_steps = 100 if kind == "layout" else 150
    prompt = table_query_tokens(cfg.decoder, B).to(dev) if kind == "table" else None

    def timed(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms / k

    def whole(px):
        if kind == "layout":
            return layout_greedy(eng, px, n_steps)[0]
        return table_greedy(eng, px, prompt, n_steps)[0]

    def e2e():
        tok = whole(x_host.to(dev, non_blocking=True))
        tok.cpu()

    for _ in range(max(3, warmup)):
        eng.encode(x)
    ms_enc = timed(lambda: eng.encode(x), max(1, steps))
    whole(x)
    k = max(1, min(steps, 2))
    ms_all = timed(lambda: whole(x), k)
    ms_e2e = timed(e2e, k)
    gflop = 326.6 if kind == "layout" else 268.6
    tf = gflop * B / (ms_enc * 1e-3) / 1e3
    res = {"metric": f"pages/sec ({kind})", "value": B * world / (ms_all * 1e-3), "unit": "pages/s", "ms_per_step": ms_all,
           "e2e": {"value": B * world / (ms_e2e * 1e-3), "unit": "pages/s", "h2d_bytes_per_step": x_host.numel() * 2,
                   "d2h_bytes_per_step": B * n_steps * (7 if kind == "layout" else 10) * 8},
           "config": {"workload": f"{kind}: {B} synthetic 768x768 pages per GPU, Swin encoder + {n_steps} greedy decoder steps",
                      "dtype": "f16"},
           "phases_ms": {"encoder": ms_enc, "decode": ms_all - ms_enc, "decode_step": (ms_all - ms_enc) / n_steps},
           "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                        "frac": tf / peaks["tf_sustained"], "alg_gflop_per_page": gflop, "scope": "Swin encoder (linear layers)"}}
    return res


def ocr_error_bench(dev, world, steps, warmup, timed):
    """SURVEY §8 f4: DistilBertForSequenceClassification (default config, fp16 = the reference's CUDA dtype) on the predictor's CUDA
    batch of 64 texts (surya/ocr_error/__init__.py:16) right-padded to 512 tokens, lengths uniform in [16, 512].  `value`: texts/s of
    the packed forward with the token plan already on the host; `e2e`: detect_errors() from host int64 ids / masks to label strings."""
    from surya_b200.config import ocr_error_default
    from surya_b200.ocr_error import B200DistilBert, build_pack_plan, detect_errors
    from surya_b200.synth import ocr_error_state_dict, ocr_error_synthetic_batch

    cfg = ocr_error_default()
    model = B200DistilBert(cfg, ocr_error_state_dict(cfg, seed=0), dtype=torch.float16, device=dev)
    n_batches, B, L = 4, 64, 512
    ids, mask = ocr_error_synthetic_batch(cfg, n_batches * B, L, seed=21, min_len=16)
    plans = [build_pack_plan(ids[i * B:(i + 1) * B].numpy(), mask[i * B:(i + 1) * B].numpy(), cfg) for i in range(n_batches)]
    n_tok = sum(p["n_tok"] for p in plans)

    def resident():
        for p in plans:
            model.forward_packed(p)

    def e2e():
        detect_errors(model, ids, mask, batch_size=B)

    for _ in range(max(1, warmup)):
        resident()
    k = max(1, min(steps, 5))
    ms = timed(resident, k) / k
    e2e()
    ms_e2e = timed(e2e, k) / k
    texts = n_batches * B * world
    flop = 2.0 * n_tok * cfg.n_layers * (4 * cfg.dim * cfg.dim + 2 * cfg.dim * cfg.hidden_dim)
    return {"metric": "texts/sec (ocr_error)", "value": texts / (ms * 1e-3), "unit": "texts/s", "ms_per_step": ms,
            "e2e": {"value": texts / (ms_e2e * 1e-3), "unit": "texts/s", "h2d_bytes_per_step": int(n_tok * 8 + n_batches * B * 8),
                    "d2h_bytes_per_step": n_batches * B * 8},
            "config": {"workload": f"ocr_error: {n_batches} batches of {B} texts, right-padded to {L}, {n_tok} real tokens (packed; pad "
                                   "positions are never computed)", "dtype": "f16"},
            "linear_tflops": flop / (ms * 1e-3) / 1e12}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the PyTorch-eager-on-GPU secondary baseline")
    ap.add_argument("--no-detection", action="store_true")
    ap.add_argument("--no-layout", action="store_true", help="skip the layout / table_rec (config 4) secondary numbers")
    ap.add_argument("--no-pipeline", action="store_true", help="skip the ocr_text pipeline (config 5) secondary number")
    ap.add_argument("--no-ocr-error", action="store_true", help="skip the ocr_error (DistilBERT) secondary number")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's tokens / scores / boxes as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        return run_reference_arm(args)
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist

    from surya_b200 import _lib
    from surya_b200.config import syn_rec
    from surya_b200.recognition import RecEngine, RecognitionRunner, build_prefill_plan, pack_rec_weights
    from surya_b200.synth import rec_state_dict, rec_synthetic_crops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise _lib.SuryaB200Error("bench.py needs a B200 (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = _peaks()
    log(f"rank {rank}/{world} on cuda:{local}")
    cfg = syn_rec()
    dtype = torch.bfloat16

    # ---- weights: rank 0 packs, NCCL broadcast to the replicas (SURVEY.md §8e)
    if rank == 0:
        weights = pack_rec_weights(rec_state_dict(cfg, seed=0), cfg, dtype, dev)
        meta = [(tuple(w.shape), str(w.dtype)) for w in weights]
    else:
        weights, meta = None, None
    if world > 1:
        box = [meta]
        dist.broadcast_object_list(box, src=0)
        meta = box[0]
        if rank != 0:
            weights = [torch.empty(s, dtype=getattr(torch, d.split(".")[-1]), device=dev) for s, d in meta]
        for w in weights:
            dist.broadcast(w, src=0)
    eng = RecEngine(cfg, None, dtype=dtype, device=dev, max_slots=B_PER_GPU + 4, s_max=256, max_patches=B_PER_GPU * 160,
                    max_tokens=B_PER_GPU * 46, packed_weights=weights)
    log(f"engine ready, workspace {eng.workspace_bytes / 1e9:.2f} GB")
    runner = RecognitionRunner(eng, batch_size=B_PER_GPU, max_tokens=MAX_TOKENS)
    crops = list(rec_synthetic_crops(B_PER_GPU, CROP_H, CROP_W, seed=1234 + rank))
    tiles, grids, seqs = runner.preprocess(crops)
    tiles_host = torch.from_numpy(np.concatenate(tiles, 0)).pin_memory()
    h2d_bytes = tiles_host.numel() * 4
    slots = eng.alloc_slots(B_PER_GPU)
    plan = build_prefill_plan(cfg, np.array(grids), seqs, slots)
    h2d_bytes += plan.ints.numel() * 4 + plan.ids.numel() * 8
    d2h_bytes = B_PER_GPU * MAX_TOKENS * (8 + 4 + 48)

    # ---- resident step: inputs in HBM, outputs stay on the device
    tiles_dev = tiles_host.to(dev)
    plan.ints = plan.ints.to(dev)
    plan.ids = plan.ids.to(dev)
    slot_t = torch.tensor(slots, dtype=torch.int32, device=dev)
    lens = torch.tensor([len(s) for s in seqs], dtype=torch.int32, device=dev)
    max_len = max(len(s) for s in seqs)
    ids_io = torch.empty(B_PER_GPU, dtype=torch.int64, device=dev)
    pos_io = torch.empty(B_PER_GPU, dtype=torch.int32, device=dev)
    hist = {"tok": torch.empty((MAX_TOKENS - 1, B_PER_GPU), dtype=torch.int64, device=dev),
            "score": torch.empty((MAX_TOKENS - 1, B_PER_GPU), dtype=torch.float32, device=dev),
            "bbox": torch.empty((MAX_TOKENS - 1, B_PER_GPU, 6), dtype=torch.int64, device=dev),
            "done": torch.empty((MAX_TOKENS - 1, B_PER_GPU), dtype=torch.uint8, device=dev)}
    from surya_b200 import shard

    last = {}

    def resident_step():
        out = eng.prefill(tiles_dev, plan)
        last["prefill"] = out
        ids_io.copy_(out["next_ids"])
        pos_io.copy_(lens)
        eng.decode_steps(ids_io, slot_t, pos_io, MAX_TOKENS - 1, hist=hist, max_pos=max_len)
        if world > 1:       # tokens, scores AND boxes of every replica, through the product's sharding helper (SURVEY.md §8e)
            shard.gather_step_results(hist["tok"], hist["score"], hist["bbox"])
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    log("inputs ready; warm-up")
    for _ in range(args.warmup):
        resident_step()
    torch.cuda.synchronize()
    log("timed region")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    ms_total = timed(resident_step, args.steps)
    launches = _lib.launch_count() - l0
    ms_step = ms_total / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["prefill"], hist)
    value = B_PER_GPU * world * args.steps / (ms_total * 1e-3)

    # ---- phase split (CUDA events, rank-local, outside the headline region)
    def prefill_only():
        eng.prefill(tiles_dev, plan)

    def decode_only():
        pos_io.copy_(lens)
        eng.decode_steps(ids_io, slot_t, pos_io, MAX_TOKENS - 1, hist=hist, max_pos=max_len)

    log(f"resident: {ms_step:.2f} ms/step -> {value:.1f} crops/s; phase split")
    ms_prefill = timed(prefill_only, 3) / 3
    ms_decode = timed(decode_only, 3) / 3
    eng.release_slots(slots)

    # ---- e2e: public API from pinned host buffers, results read back to the host
    def e2e_step():
        runner.run_preprocessed(tiles_host, grids, seqs, fixed_steps=True)

    log(f"prefill {ms_prefill:.2f} ms, decode {ms_decode:.2f} ms; e2e")
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    ms_e2e_total = timed(e2e_step, max(1, min(args.steps, 3)))
    e2e_n = max(1, min(args.steps, 3))
    e2e_value = B_PER_GPU * world * e2e_n / (ms_e2e_total * 1e-3)
    # ---- e2e from uint8 crops (SURVEY §8 f2): the preprocessing of SuryaOCRProcessor inside the timed region, on the device
    # (sb_rec_preprocess; 3 B / pixel up) and, for comparison, through the OpenCV thread pool on the host
    from_crops = None
    try:
        if world > 1:
            raise RuntimeError("single-GPU diagnostic (skipped under torchrun)")

        def crops_device():
            runner.run(crops, fixed_steps=True, preprocess="device")

        def crops_host():
            runner.run(crops, fixed_steps=True, preprocess="host")

        crops_device()
        ms_cd = timed(crops_device, e2e_n) / e2e_n
        crops_host()
        ms_ch = timed(crops_host, 1)
        from_crops = {"value": B_PER_GPU * world / (ms_cd * 1e-3), "unit": "crops/s", "ms_per_step": ms_cd,
                      "h2d_bytes_per_step": int(sum(c.size for c in crops)) + B_PER_GPU * 36, "d2h_bytes_per_step": d2h_bytes,
                      "api": "RecognitionRunner.run(uint8 crops, preprocess='device'): pack + upload + sb_rec_preprocess (Lanczos4 "
                             "scale_to_fit, cubic to x28, normalise, tile) + prefill + 127 decode steps",
                      "host_preprocess": {"value": B_PER_GPU * world / (ms_ch * 1e-3), "unit": "crops/s", "ms_per_step": ms_ch,
                                          "api": "same call with preprocess='host' (OpenCV thread pool, fp32 tiles up)"}}
        log(f"e2e from uint8 crops: device preprocessing {from_crops['value']:.1f} crops/s, host preprocessing "
            f"{from_crops['host_preprocess']['value']:.1f} crops/s")
    except Exception as e:      # noqa: BLE001
        from_crops = None if world > 1 else {"error": f"{type(e).__name__}: {e}"}
        if world == 1:
            log(f"e2e from crops failed: {from_crops['error']}")
    ocr_err = None
    if not args.no_ocr_error and world == 1:
        try:
            ocr_err = ocr_error_bench(dev, world, args.steps, args.warmup, timed)
            log(f"ocr_error: {ocr_err['value']:.0f} texts/s resident, {ocr_err['e2e']['value']:.0f} e2e")
        except Exception as e:      # noqa: BLE001
            ocr_err = {"error": f"{type(e).__name__}: {e}"}
            log(f"ocr_error failed: {ocr_err['error']}")
    # secondary sections must never cost the headline line: a failure is reported inside the JSON instead (all ranks take the
    # same path because the inputs are identical, so the collectives inside stay matched)
    det = None
    if not args.no_detection:
        log("detection (secondary metric)")
        try:
            det = detection_bench(dev, peaks, world, args.steps, args.warmup)
            log(f"detection: {det['value']:.1f} pages/s resident, {det['e2e']['value']:.1f} e2e")
        except Exception as e:      # noqa: BLE001
            det = {"error": f"{type(e).__name__}: {e}"}
            log(f"detection failed: {det['error']}")
    lay = None
    if not args.no_layout:
        lay = {}
        for kind in ("layout", "table"):
            log(f"{kind} (config 4)")
            try:
                lay[kind] = layout_bench(dev, peaks, world, kind, args.steps, args.warmup)
                log(f"{kind}: {lay[kind]['value']:.1f} pages/s (encoder {lay[kind]['phases_ms']['encoder']:.2f} ms, "
                    f"decode step {lay[kind]['phases_ms']['decode_step']:.3f} ms)")
            except Exception as e:      # noqa: BLE001
                lay[kind] = {"error": f"{type(e).__name__}: {e}"}
                log(f"{kind} failed: {lay[kind]['error']}")
    pipe = None
    if not args.no_pipeline:
        log("ocr_text pipeline (config 5)")
        try:
            pipe = pipeline_bench(dev, world, rank, eng)
            log(f"pipeline: {pipe['value']:.1f} pages/s end to end, {pipe['lines_total']} lines")
        except Exception as e:      # noqa: BLE001
            pipe = {"error": f"{type(e).__name__}: {e}"}
            log(f"pipeline failed: {pipe['error']}")
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        log(f"e2e {e2e_value:.1f} crops/s; roofline replay")
        try:
            roof, gemm_ms = decode_gemm_roofline(eng, peaks)
            roof["share_of_step"] = gemm_ms * (MAX_TOKENS - 1) / ms_step          # of the whole step (prefill + 127 decode steps)
            roof["share_of_decode_step"] = gemm_ms / (ms_decode / (MAX_TOKENS - 1))
            roof["share_note"] = ("ncu's launch list gives these launches 0.81 of one decode step's summed kernel time "
                                  "(profiles/decode_gemm_traffic.json); in the graph ~0.10 ms of the 0.87 ms step is launch-to-launch "
                                  "gap, which a sum of kernel durations does not contain")
        except Exception as e:      # noqa: BLE001
            roof = {"error": f"{type(e).__name__}: {e}"}
        # whole-step algorithmic bounds (SURVEY.md §8d) for context
        alg = {"decode_bytes_per_step_gb": 1.02, "decode_hbm_ms_at_peak": 1.02e9 * (MAX_TOKENS - 1) / (peaks["hbm_gbs"] * 1e9) * 1e3,
               "prefill_gflop_per_crop": 53.26 + 19.0, "prefill_tensor_ms_at_peak": (53.26 + 19.0) * B_PER_GPU / (peaks["tf_sustained"] * 1e3) * 1e3}
        eager = None
        if not args.no_eager_baseline:
            log("gpu_eager_baseline: reference algorithm in PyTorch eager on this GPU")
            try:
                eager = gpu_eager_baseline(dev)
                log(f"gpu_eager_baseline: recognition {eager['recognition']['value']:.1f} crops/s, detection "
                    f"{eager['detection']['value']:.1f} pages/s")
            except Exception as e:      # noqa: BLE001
                eager = {"error": f"{type(e).__name__}: {e}"}
                torch.cuda.empty_cache()
        cpu = None
        if not args.no_cpu_baseline:
            log(f"cpu_baseline: oracle port on {host_threads()} threads")
            try:
                cpu, _ = cpu_baseline_run(2)
            except Exception as e:      # noqa: BLE001
                cpu = {"error": f"{type(e).__name__}: {e}"}
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": "crops/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": _config(world),
            "e2e": {"value": e2e_value, "unit": "crops/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "api": "surya_b200.recognition.RecognitionRunner.run_preprocessed (host tiles -> tokens/scores/boxes)"},
            "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu, "gpu_eager_baseline": eager, "clocks": clocks,
            "phases_ms": {"prefill(vision+decoder)": ms_prefill, f"decode x{MAX_TOKENS - 1}": ms_decode,
                          "decode_step": ms_decode / (MAX_TOKENS - 1)},
            "algorithmic": alg, "engine_workspace_gb": eng.workspace_bytes / 1e9, "detection": det,
            "layout": lay["layout"] if lay else None, "table_rec": lay["table"] if lay else None, "ocr_pipeline": pipe,
            "e2e_from_crops": from_crops, "ocr_error": ocr_err,
        }))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
