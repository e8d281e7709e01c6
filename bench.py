#!/usr/bin/env python
"""bench.py -- real-time factor of the Qwen3-ASR hot path on B200 (BASELINE.json metric).

A "step" = one pass of the hot path (transcribe() steps 2-8, /root/reference/src/inference.rs:94-200:
f32 samples -> mel -> encoder -> prefill -> greedy decode -> token ids) over one batch of synthetic
30 s / 16 kHz clips.  Default workload `b1`: ONE clip per GPU (BASELINE.json configs[1]; weak scaling over
--gpus).  Synthetic weights of the Qwen3-ASR-0.6B architecture never emit EOS, so the decode length is fixed
at --new-tokens (SURVEY.md section 8d "fixed 128 new tokens").

  value : whole-job RTF with the samples already resident in HBM (no H2D in the timed region)
  e2e   : same metric through the public host-buffer API (pinned H2D of the samples and D2H of the
          ids inside the timed region, plus the NCCL gather of ids when N > 1)
  roofline : the decode step (HBM-bound): algorithmic bytes / CUDA-event duration vs measured peak
  cpu_baseline : the oracle (CPU restatement of the reference's tch-CPU path) timed on this box
  extra : (N = 1 only) the other BASELINE.json configs on one GPU, each with its own roofline:
          b8 (north_star "batch 8 x 30 s"), decode512 (configs[4] per GPU: 16 sequences, 512-token KV),
          enc64 (configs[2]: encoder GEMM TFLOP/s at batch 64); `--workload 1p7b` adds configs[3]'s model.

--workload {all,b1,b8,decode512,enc64,1p7b}: `all` (default) = b1 headline + extras; any other value = b1 headline
plus only that extra.  --impl reference times only the CPU restatement (the Rust reference cannot be built: no cargo).

--steps K: each timed pass (e2e, then value) runs exactly K steps.
--dump-outputs DIR: after the timed steps, write what the last one returned to its caller as DIR/ids.npy (float64
[clips, --new-tokens], -1 past a clip's end; on N > 1 the ids of every rank's clip, as the gather delivers them).
Weights and clips are seeded, so the same arguments give the same inputs and two builds can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark may run from a read-only tree and must leave it untouched

CLIP_SECONDS = 30.0
METRIC = "real-time factor (audio-sec/wall-sec) Qwen3-ASR-0.6B 30s clips"     # identical in both arms
ENC_GFLOP_PER_CLIP = 270.7      # SURVEY.md section 8d: conv 131.6 + 18 layers 135.26 + windowed attention 2.49 + head 1.34
PROMPT_TOKENS_30S = 390 + 15    # audio tokens of a 30 s clip + fixed prompt tokens


def load_traffic():
    """dram bytes per decode-step launch from the newest committed `ncu --set full` capture (profiles/), or None."""
    for name in ("r02_decode_step_ncu_summary.json", "r01_decode_step_ncu_summary.json"):
        p = os.path.join(ROOT, "profiles", name)
        try:
            with open(p) as f:
                d = json.load(f)
            return float(d["dram_bytes_read"] + d["dram_bytes_write"]), f"profiles/{name} (ncu --set full, 1 launch)"
        except (OSError, KeyError, ValueError):
            continue
    return None, None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", 1389.3)), "measured"
    return 6650.0, 1400.0, "fallback"


def decode_step_bytes(cfg, ctx_tokens: float, batch: int = 1) -> float:
    """Algorithmic HBM bytes of one decoder forward step (SURVEY.md section 8d): every weight once
    (bf16) + the KV cache of `ctx_tokens` tokens (fp32 in parity mode) + the KV append."""
    t = cfg.text
    q_dim, kv_dim = t.num_attention_heads * t.head_dim, t.num_key_value_heads * t.head_dim
    per_layer = (q_dim + 2 * kv_dim) * t.hidden_size + t.hidden_size * q_dim + 3 * t.intermediate_size * t.hidden_size
    weights = (t.num_hidden_layers * per_layer + t.vocab_size * t.hidden_size) * 2
    kv = batch * t.num_hidden_layers * 2 * kv_dim * (ctx_tokens + 1) * 4
    return float(weights + kv)


class ClockSampler:
    def __init__(self, device: int):
        self.device = device
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                       "-i", str(self.device), "-lms", "200"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def host_info():
    """What the CPU arm ran on (the round-1 CPU numbers differed 5.6x between two boxes with the same core count)."""
    model = None
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    try:
        aff = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        aff = None
    try:
        load = os.getloadavg()[0]
    except OSError:
        load = None
    return {"cpu_model": model, "os_cpu_count": os.cpu_count(), "affinity": aff, "loadavg_1m": load}


def cpu_threads_setup():
    import torch
    if os.environ.get("OMP_NUM_THREADS") == "1" and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        # torchrun pins OMP_NUM_THREADS=1 per rank; the CPU arm runs on rank 0 alone and may use the host's cores
        try:
            n = len(os.sched_getaffinity(0))
        except (AttributeError, OSError):
            n = os.cpu_count() or 1
        torch.set_num_threads(max(1, min(n, 64)))
    return torch.get_num_threads()


def dump_outputs(out_dir: str, ids, width: int) -> None:
    """Token ids per clip as DIR/ids.npy: float64 (every token id is exact), [clips, width], -1 past a clip's end."""
    import numpy as np
    a = np.full((len(ids), width), -1.0, dtype=np.float64)
    for i, row in enumerate(ids):
        a[i, :len(row)] = row
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "ids.npy"), a)


_ORACLE = {}


def cpu_reference_run(new_tokens: int, reps: int):
    """The oracle timed on the host cores: one 30 s clip, `new_tokens` greedy tokens, batch 1,
    exactly as the reference would run it (lm_head over all prefill rows included)."""
    from oracle import oracle as O
    from qwen3_asr_rs_b200 import synth
    threads = cpu_threads_setup()
    if "model" not in _ORACLE:
        cfg = O.cfg_0p6b()
        _ORACLE["model"] = O.OracleModel(cfg, synth.make_weights(cfg, 1))
        _ORACLE["clip"] = synth.make_clip(0, CLIP_SECONDS)
    times, last = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        last = O.transcribe_ids(_ORACLE["model"], _ORACLE["clip"], max_new_tokens=new_tokens)
        times.append(time.perf_counter() - t0)
    return times, last, threads


def base_config(world: int, new_tokens: int):
    return {"workload": "Qwen3-ASR-0.6B, batch=1 per GPU, single 30 s 16 kHz clip, greedy decode",
            "clips_per_gpu": 1, "clip_seconds": CLIP_SECONDS, "new_tokens": new_tokens,
            "weights": "synthetic bf16 (seed 1), Qwen3-ASR-0.6B architecture", "activations": "fp32-exact (bf16x3 split / fp32)",
            "l2": "inputs larger than L2: 1.19 GB of weights streamed every decode step",
            "parallelism": f"dp{world}"}


def reference_arm(args, K, W):
    """--impl reference: the CPU restatement of the reference's path, same metric / config / warm-up as our arm.
    Each step is the whole workload step (one 30 s clip, --new-tokens tokens) unless that cannot finish K + W steps
    in ~6 minutes on this host; then a step is the same clip with fewer new tokens and `value` is completed with this
    run's measured per-token time (flagged `extrapolated`)."""
    info0 = host_info()
    t0 = time.perf_counter()
    times_w, _, threads = cpu_reference_run(args.new_tokens, 1)          # warm-up step 1 = calibration
    t_full = times_w[0]
    budget = float(os.environ.get("ASRB_REF_BUDGET_S", "360"))
    n_tok, extrapolated = args.new_tokens, False
    if t_full * (K + W - 1) > budget and args.new_tokens > 16:
        n_tok, extrapolated = 16, True
    for _ in range(max(0, W - 1)):
        cpu_reference_run(n_tok, 1)
    times, last, _ = cpu_reference_run(n_tok, K)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [last.ids], args.new_tokens)
    T = sum(times) / K
    per_tok = None
    if extrapolated:
        t16 = T
        per_tok = max(0.0, (t_full - t16) / (args.new_tokens - n_tok))
        T = t16 + per_tok * (args.new_tokens - n_tok)
    v = CLIP_SECONDS / T
    info1 = host_info()
    sample = (f"{K} x one 30 s clip, {n_tok} new tokens per step" +
              (f" (+ {args.new_tokens - n_tok} tokens at this run's measured {1e3 * per_tok:.1f} ms/token)" if extrapolated else "") +
              ", PyTorch-CPU fp32 restatement of the reference's tch-CPU path (Rust toolchain absent)")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "x realtime",
            "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": 1e3 * T,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": base_config(max(1, int(os.environ.get("WORLD_SIZE", "1"))), args.new_tokens),
            "cpu_baseline": {"value": v, "unit": "x realtime", "cores": threads, "kind": "port", "sample": sample,
                             "extrapolated": extrapolated, "torch_threads": threads, "host": info0,
                             "loadavg_1m_after": info1["loadavg_1m"], "wall_s": time.perf_counter() - t0},
            "e2e": {"value": v, "unit": "x realtime", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------
# extras: the other BASELINE.json configs on one GPU (never part of the headline timing)
# ------------------------------------------------------------------------------------------------------
def extra_batch_decode(eng, cfg, synth, B, new_tokens, hbm_peak, label):
    clips = [synth.make_clip(i, CLIP_SECONDS) for i in range(B)]
    for _ in range(2):
        r = eng.transcribe_ids(clips, max_new_tokens=new_tokens)
    steps = max(r.decode_steps, 1)
    us = 1e3 * r.stage_ms["decode"] / steps
    ctx = PROMPT_TOKENS_30S + (new_tokens - 1) / 2.0
    by = decode_step_bytes(cfg, ctx, B)
    return {"workload": label, "batch": B, "new_tokens": new_tokens, "avg_kv_tokens": ctx,
            "rtf": CLIP_SECONDS * B / (r.stage_ms["total"] / 1e3), "stage_ms": {k: round(v, 3) for k, v in r.stage_ms.items()},
            "decode_us_per_step": us, "decode_tokens_per_s": B * 1e6 / us,
            "roofline": {"kernel": f"decoder forward step (batch {B})", "bound": "hbm", "bytes_per_launch": by,
                         "achieved": by / us / 1e3, "peak": hbm_peak, "unit": "GB/s", "frac": by / us / 1e3 / hbm_peak},
            "stats": eng.stats()}


def extra_encoder(eng, synth, B, tf_peak):
    clips = [synth.make_clip(i, CLIP_SECONDS) for i in range(B)]
    for _ in range(2):
        r = eng.transcribe_ids(clips, max_new_tokens=2)
    enc_ms = r.stage_ms["encoder"]
    tf = ENC_GFLOP_PER_CLIP * B / enc_ms
    return {"workload": f"Qwen3-ASR-0.6B, batch={B} synthetic 30 s clips, 1xB200 (encoder GEMM roofline)", "batch": B,
            "encoder_ms": enc_ms, "mel_ms": r.stage_ms["mel"], "prefill_ms": r.stage_ms["prefill"],
            "roofline": {"kernel": "audio encoder (conv stem + 18 layers + head)", "bound": "tensor",
                         "flops_per_launch": ENC_GFLOP_PER_CLIP * 1e9 * B, "achieved": tf, "peak": tf_peak, "unit": "TFLOP/s",
                         "frac": tf / tf_peak, "note": "algorithmic FLOPs; every fp32-exact GEMM issues 3 bf16 MMAs per product"},
            "stats": eng.stats()}


def extra_1p7b(synth, device, new_tokens, hbm_peak):
    from qwen3_asr_rs_b200 import AsrInference, config_1p7b
    cfg = config_1p7b()
    eng = AsrInference.from_weights(cfg, synth.make_weights(cfg, 3), device=device)
    try:
        clip = synth.make_clip(0, CLIP_SECONDS)
        for _ in range(2):
            r = eng.transcribe_ids([clip], max_new_tokens=new_tokens)
        steps = max(r.decode_steps, 1)
        us = 1e3 * r.stage_ms["decode"] / steps
        by = decode_step_bytes(cfg, PROMPT_TOKENS_30S + (new_tokens - 1) / 2.0, 1)
        return {"workload": "Qwen3-ASR-1.7B (dims as recalled in SURVEY.md section 8), batch=1, 30 s clip", "new_tokens": new_tokens,
                "rtf": CLIP_SECONDS / (r.stage_ms["total"] / 1e3), "stage_ms": {k: round(v, 3) for k, v in r.stage_ms.items()},
                "decode_us_per_step": us,
                "roofline": {"kernel": "decoder forward step (batch 1)", "bound": "hbm", "bytes_per_launch": by,
                             "achieved": by / us / 1e3, "peak": hbm_peak, "unit": "GB/s", "frac": by / us / 1e3 / hbm_peak},
                "stats": eng.stats()}
    finally:
        eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--new-tokens", type=int, default=128)
    ap.add_argument("--workload", default="all", choices=["all", "b1", "b8", "decode512", "enc64", "1p7b"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--decode", default=None, choices=[None, "mega", "phases"])
    ap.add_argument("--gemm", default=None, choices=[None, "tc", "simt"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the ids returned by the last timed step to DIR/ids.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = args.steps, max(args.warmup, 3)       # both arms: W >= 3 warm-up steps
    config = base_config(world, args.new_tokens)

    if args.impl == "reference":
        if rank != 0:
            return
        reference_arm(args, K, W)
        return

    import torch
    from qwen3_asr_rs_b200 import AsrInference, config_0p6b, parallel, synth

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    cfg = config_0p6b()
    weights = synth.make_weights(cfg, 1)
    eng = AsrInference.from_weights(cfg, weights, device=local_rank)
    del weights
    if args.decode:
        eng.set_option("decode", args.decode)
    if args.gemm:
        eng.set_option("gemm", args.gemm)
    clip = synth.make_clip(rank, CLIP_SECONDS)
    dev = torch.device("cuda", local_rank)
    gather = parallel.IdsGather(world, world, args.new_tokens, dev) if dist is not None else None

    def one_step():
        """-> (per-step result, the ids of every clip of the job as the caller receives them)"""
        r = eng.transcribe_ids([clip], max_new_tokens=args.new_tokens)
        if gather is not None:   # the path's only collective: gather of decoded ids (NCCL over NVLink, device buffers)
            return r, gather(eng)
        return r, r.ids

    for _ in range(W):
        last, _ = one_step()
    # ---- e2e: host buffers in, ids out ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    try:
        barrier()
        t0 = time.perf_counter()
        stage = {}
        launches = 0
        dec_ms, dec_steps = 0.0, 0
        for _ in range(K):
            last, _ = one_step()
            for k, v in last.stage_ms.items():
                stage[k] = stage.get(k, 0.0) + v / K
            launches = last.kernels_launched
            dec_ms += last.stage_ms["decode"]; dec_steps += last.decode_steps
        barrier()
        t_e2e = time.perf_counter() - t0
        # ---- value: samples resident in HBM ----
        eng.set_option("resident", "1")
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            last, out_ids = one_step()
        barrier()
        t_val = time.perf_counter() - t0
    finally:                # never leave the nvidia-smi sampler running
        clocks = sampler.stop() if rank == 0 else None
    eng.set_option("resident", "0")
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out_ids, args.new_tokens)
    if dist is not None:
        tt = torch.tensor([t_e2e, t_val], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_e2e, t_val = float(tt[0]), float(tt[1])
    ids = last.ids[0]
    stats = eng.stats()
    if rank == 0:
        audio_total = CLIP_SECONDS * world * K
        value, e2e = audio_total / t_val, audio_total / t_e2e
        hbm_peak, tf_peak, peak_kind = load_peaks()
        ctx_avg = PROMPT_TOKENS_30S + (args.new_tokens - 1) / 2.0
        step_bytes = decode_step_bytes(cfg, ctx_avg)
        step_s = (dec_ms / 1e3) / max(dec_steps, 1)
        achieved = step_bytes / step_s / 1e9
        traffic, traffic_src = load_traffic()
        line = {"metric": METRIC, "value": value, "unit": "x realtime",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": 1e3 * t_val / K, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32 (bf16 weights, fp32-exact activations)", "data": "synthetic",
                "config": config,
                "e2e": {"value": e2e, "unit": "x realtime", "h2d_bytes_per_step": int(clip.nbytes),
                        "d2h_bytes_per_step": int(4 * (args.new_tokens + 1)), "ms_per_step": 1e3 * t_e2e / K},
                "gpu_launches": int(launches) * K * 2 + 0,
                "stage_ms": {k: round(v, 4) for k, v in stage.items()},
                "decode": {"steps_per_clip": dec_steps // K, "us_per_step": 1e6 * step_s, "tokens": len(ids)},
                "roofline": {"kernel": "decoder forward step (batch 1)", "bound": "hbm", "achieved": achieved, "peak": hbm_peak,
                             "unit": "GB/s", "frac": achieved / hbm_peak, "peak_kind": peak_kind,
                             "bytes_per_launch": step_bytes, "traffic": traffic, "traffic_source": traffic_src},
                "path_stats": stats,
                "clocks": clocks}
        # silent fallbacks are errors: the headline must have run on the fused decode step and tcgen05 GEMMs only
        if not args.decode and not args.gemm:
            assert stats.get("decode_phase_steps", 0) == 0 and stats.get("gemm_simt_fallbacks", 0) == 0, stats
        if world == 1:
            extra = {}
            want = args.workload
            try:
                if want in ("all", "b8"):
                    extra["b8"] = extra_batch_decode(eng, cfg, synth, 8, args.new_tokens, hbm_peak,
                                                     "Qwen3-ASR-0.6B, batch=8 x 30 s clips, 1xB200 (north_star batch)")
                if want in ("all", "decode512"):
                    # 16 sequences per GPU (= BASELINE configs[4]'s 128 / 8 GPUs); 215 new tokens put the AVERAGE KV length at 512
                    extra["decode512"] = extra_batch_decode(eng, cfg, synth, 16, 215, hbm_peak,
                                                            "Qwen3-ASR-0.6B decode, 16 sequences per GPU, 512-token KV cache (BASELINE configs[4] per GPU)")
                if want in ("all", "enc64"):
                    extra["enc64"] = extra_encoder(eng, synth, 64, tf_peak)
            except Exception as e:          # an extra must never take the headline down with it
                extra["error"] = repr(e)
            line["extra"] = extra
        if world == 1 and not args.no_cpu_baseline:
            times, ref, threads = cpu_reference_run(args.new_tokens, 1)
            line["cpu_baseline"] = {"value": CLIP_SECONDS / times[0], "unit": "x realtime", "cores": threads, "kind": "port",
                                    "sample": f"one 30 s clip, {args.new_tokens} new tokens (the whole step), PyTorch-CPU fp32 "
                                              "restatement of the reference's tch-CPU path",
                                    "torch_threads": threads, "host": host_info(),
                                    "ids_match_gpu": ref.ids == ids}
    eng.close()
    if rank == 0 and world == 1 and args.workload == "1p7b":
        try:
            line["extra"]["1p7b"] = extra_1p7b(synth, local_rank, 64, load_peaks()[0])
        except Exception as e:
            line["extra"]["1p7b_error"] = repr(e)
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
