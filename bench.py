#!/usr/bin/env python
"""Headline benchmark: audio-seconds generated per wall-second (and RTF) for Chatterbox 0.5B on 256-utterance
synthetic batches, one process per GPU (BASELINE.json metric; SURVEY.md 8d config 3).

    python bench.py --gpus N --steps K --warmup W            # this engine (torchrun launches N ranks)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU algorithm timed on the host cores,
                                                             # each step one bounded sample of the same workload

A "step" = one full pass of the hot path over one batch: T3 prefill + AR decode with CFG -> token clean-up ->
flow encoder -> 10-step CFM with CFG -> HiFT vocoder, for 256 mixed-length utterances per GPU (weak scaling:
every rank owns its own 256 utterances; the only collective is the broadcast of the voice conditionals).
Weights are seeded random-init tensors of the exact reference architecture (no checkpoints / network here);
utterance length is set by per-utterance max_new_tokens ~ U(75, 1000) as SURVEY.md 8d prescribes.

Order of a run (engine arm):
  1. W warm-up steps, then K timed steps with inputs resident on the device -- NO per-kernel timers inside (`value`);
  2. `e2e`: the public batch API with host token ids in, waveforms back in pinned host memory;
  3. profiling passes OUTSIDE the timed region: CUDA-event timers around one kernel class per pass (gemm_tc, attn_tc,
     paged attention) -> `roofline` (the class with the largest share) and `config.kernel_rooflines`;
  4. the other BASELINE configs, one warm + one timed pass each, reported under `config`:
     strong_256 (N > 1: 256 utterances TOTAL, LPT-sharded over the ranks), mtl_256 (config 4, multilingual vocabulary,
     256 total), turbo_512 (config 5, Turbo 350M, 512 total, 2-step meanflow), b1_latency (config 2);
  5. `cpu_baseline` (rank 0, N = 1 only): k = 4 utterances of the batch (sorted indices 0 / 85 / 170 / 255) through the
     reference's CPU path (the oracle port of the reference algorithm).
  --dump-outputs DIR: after the timed steps, the waveforms of the last one (see dump_outputs) for output comparison.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
_T0 = time.time()


def log(*a):
    if os.environ.get("CBX_BENCH_VERBOSE", "1") != "0" and int(os.environ.get("RANK", 0)) == 0:
        print(f"[bench {time.time() - _T0:7.1f}s]", *a, file=sys.stderr, flush=True)

METRIC = "audio_seconds_per_second"
WORKLOAD = "Chatterbox 0.5B en, batch=256 mixed-length utterances per GPU, CFG, 10-step CFM, paged bf16 KV"
UNIT = "audio-s/s"
SEED = 20260922
N_PROMPT = 250                      # S3Gen prompt tokens of the synthetic voice (10 s)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


def make_workload(batch, seed, rank, budget_max=1000, vocab_lo=1, vocab_hi=255):
    """SURVEY.md 8d config 3: N_text ~ randint(16,160), ids randint(1,255), N ~ randint(75,1000)."""
    g = torch.Generator().manual_seed(seed + 7919 * rank)
    n_text = torch.randint(16, 160, (batch,), generator=g)
    texts = [torch.randint(vocab_lo, vocab_hi, (int(n),), generator=g) for n in n_text]
    budgets = torch.randint(min(75, budget_max - 1), budget_max, (batch,), generator=g).tolist()
    return texts, budgets


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def host_threads():
    """Threads the CPU arm may really use: scheduler affinity and cgroup quota, not the raw core count of the host."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = min(n, max(1, int(float(q[0]) / float(q[1]))))
    except Exception:
        pass
    return max(1, min(n, 64))


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# ------------------------------------------------------------------------------------------------ CPU reference arm
class CpuReference:
    """The reference's CPU path for one utterance at a time (the reference is batch-1): T3.inference (CFG pair, sampler
    defaults of generate(): T 0.8, min_p 0.05, rep 1.2, cfg 0.5) -> token clean-up -> flow (10 NFE) -> HiFT, run by the
    oracle restatement of the same algorithm (kind = 'port')."""

    def __init__(self, threads=None):
        from oracle import weights as W
        from oracle.t3_ref import T3Oracle
        from oracle.flow_ref import FlowOracle
        from oracle.hift_ref import HiFTOracle
        self.threads = threads or host_threads()
        torch.set_num_threads(self.threads)
        self.W = W
        self.c3, self.cg = W.make_conds(1234)
        self.kind = "port"
        self.t3 = T3Oracle(W.make_t3_weights(0))
        self.flow = FlowOracle(W.make_flow_weights(0))
        self.hift = HiFTOracle(W.make_hift_weights(0))

    def utterance(self, text, budget, seed=0):
        """-> (audio_seconds, wall_seconds, split)"""
        tt = F.pad(F.pad(text.reshape(-1).long(), (1, 0), value=255), (0, 1), value=0)
        tt = torch.stack([tt, tt])
        torch.manual_seed(seed)
        t0 = time.perf_counter()
        toks = self.t3.inference(self.c3, tt, int(budget), temperature=0.8, top_p=1.0, min_p=0.05, repetition_penalty=1.2,
                                 cfg_weight=0.5)
        t1 = time.perf_counter()
        sp = toks[0]
        eos = (sp == 6562).nonzero()
        if len(eos):
            sp = sp[:int(eos[0])]
        sp = sp[sp < 6561]
        mel = self.flow.inference(sp, self.cg, 10)
        t2 = time.perf_counter()
        self.hift.inference(mel)
        t3 = time.perf_counter()
        return sp.numel() / 25.0, t3 - t0, dict(t3_s=round(t1 - t0, 2), flow_s=round(t2 - t1, 2), hift_s=round(t3 - t2, 2),
                                                tokens=int(sp.numel()), n_text=int(text.numel()))


def cpu_baseline_k4(texts, budgets):
    """SURVEY.md 8d / BASELINE.md 3: the utterances at indices 0 / 85 / 170 / 255 of the length-sorted batch, sequentially."""
    ref = CpuReference()
    order = sorted(range(len(budgets)), key=lambda b: budgets[b])
    k = min(4, len(order))
    idx = [order[int(round(i * (len(order) - 1) / max(1, k - 1)))] for i in range(k)] if k > 1 else [order[0]]
    audio = wall = 0.0
    per = []
    for i in idx:
        a, w, split = ref.utterance(texts[i], budgets[i], seed=i)
        audio += a; wall += w
        per.append(split)
        log(f"cpu baseline utt {i}: {split}")
    n = len(budgets)
    return {"value": audio / wall, "unit": UNIT, "cores": ref.threads, "kind": ref.kind, "cpu_model": cpu_model(),
            "sample": f"k={k} utterances of the bench batch (length-sorted indices {[order.index(i) for i in idx]}), sequential, "
                      "bench texts/budgets, sampler defaults, 10 NFE, HiFT",
            "wall_s": round(wall, 1), "audio_s": round(audio, 1),
            "extrapolated_batch_wall_s": round(wall * n / k, 1), "per_utterance": per}


def run_reference(args, rank, world):
    if rank != 0:
        return
    ref = CpuReference()
    texts, budgets = make_workload(args.batch, SEED, 0, args.budget_max)
    i = min(range(len(budgets)), key=lambda b: budgets[b])           # the shortest utterance of the batch: a bounded sample
    sample = (f"1 utterance per step: the shortest of the bench batch (index {i}: {int(texts[i].numel())} text tokens, budget "
              f"{budgets[i]} speech tokens, CFG pair, 250-token voice prompt, 10 NFE, HiFT)")
    for _ in range(max(1, args.warmup) if args.warmup else 0):
        ref.utterance(texts[i], budgets[i], seed=i)
    audio = wall = 0.0
    for _ in range(args.steps):
        a, w, split = ref.utterance(texts[i], budgets[i], seed=i)
        audio += a
        wall += w
    v = audio / wall
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * wall / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "rtf": wall / audio,
            "config": {"workload": WORKLOAD, "arm": "CPU oracle port of the reference algorithm (fp32, torch CPU ops in the reference's "
                                                    "order), bounded sample of the workload: one utterance per step",
                       "sample": sample, "split_s": split, "cpu_model": cpu_model()},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": ref.threads, "kind": ref.kind, "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ roofline models
def stage_work(texts, lens, n_layers=30, cfg_rows=2, nfe=10, prompt=N_PROMPT):
    """Algorithmic work of one pass (BASELINE.md 4) given the generated lengths."""
    n = np.asarray(lens, dtype=np.float64)
    s0 = np.asarray([int(t.numel()) for t in texts], dtype=np.float64) + 38.0
    # T3: weights once per decode step + KV read per row and step + KV write; prefill is tensor work
    steps = float(n.max()) if len(n) else 0.0
    kv_tok = 122880.0 * n_layers / 30.0
    t3_bytes = steps * 1.0234e9 * n_layers / 30.0 + cfg_rows * float((s0 * n + n * (n + 1) / 2).sum()) * kv_tok + cfg_rows * float(n.sum()) * kv_tok
    nn = n + prompt
    T = 2.0 * nn
    flow_flops = float((113.2e6 * nn + 90.1e3 * nn * nn).sum()) + nfe * cfg_rows * float((T * (132161536.0 + 114688.0 * T)).sum())
    frames = float((2.0 * n).sum())
    return dict(t3_bytes=t3_bytes, flow_flops=flow_flops, hift_flops=612.3e6 * frames, hift_bytes=0.30e6 * frames, frames=frames)


DUMP_BYTES = 64_000_000


def dump_sample(n_utts, budget_max):
    """Utterances whose whole waveforms --dump-outputs writes: a fixed, seeded subset, as many as fit in DUMP_BYTES at the
    longest possible waveform (960 float32 samples per speech token), less 1 MB for the lengths and the file headers."""
    k = max(1, min(n_utts, (DUMP_BYTES - 1_000_000) // (960 * 4 * budget_max)))
    return sorted(torch.randperm(n_utts, generator=torch.Generator().manual_seed(SEED))[:k].tolist())


def dump_outputs(out_dir, wavs, budget_max):
    """What generate_batch returned in the last timed step: wav_lengths.npy (float64 [B], samples of every waveform) and
    wav_<b>.npy (float32) for the utterances of dump_sample()."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "wav_lengths.npy"), np.array([w.numel() for w in wavs], dtype=np.float64))
    for b in dump_sample(len(wavs), budget_max):
        np.save(os.path.join(out_dir, f"wav_{b:03d}.npy"), wavs[b].detach().float().cpu().numpy())
    log(f"wrote the last timed step's outputs to {out_dir}")


# ------------------------------------------------------------------------------------------------ this engine
def run_engine(args, rank, world, local_rank):
    import torch.distributed as dist
    from oracle import weights as W            # only the seeded synthetic checkpoint generator + cpu_baseline leg
    from chatterbox_b200 import ChatterboxTTS, Conditionals, T3, T3Cond, S3Gen, Engine
    from chatterbox_b200.dist import broadcast_conditionals, shard_utterances, utterance_cost
    torch.cuda.set_device(local_rank)
    torch.set_num_threads(max(1, host_threads() // max(1, world)))     # host-side weight synthesis: do not oversubscribe
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    hbm_peak, tf_peak, peak_src = load_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allsum(x):
        t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t)
        return float(t[0])

    def allmax(x):
        t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def timed(fn, steps):
        """K steps between barrier + synchronize, CUDA events on the launching stream, max over ranks."""
        tm_all = []
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            tm = {}
            fn(tm)
            tm_all.append(tm)
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        return allmax(e0.elapsed_time(e1)), allmax(wall), tm_all

    # ---- model + voice (rank 0 owns the voice, NCCL broadcast: the north_star's "speaker-embedding broadcast")
    eng = Engine(local_rank)
    t3 = T3(eng, W.make_t3_weights(0))
    s3 = S3Gen(eng, W.make_flow_weights(0), W.make_hift_weights(0))
    c3, cg = W.make_conds(1234) if rank == 0 else (None, None)
    c3, cg = broadcast_conditionals(c3, cg, torch.device("cuda", local_rank), src=0)
    tts = ChatterboxTTS(t3, s3, None, f"cuda:{local_rank}", Conditionals(T3Cond(**c3), cg))
    texts, budgets = make_workload(args.batch, SEED, rank, args.budget_max)
    log(f"models loaded; batch={args.batch} sum_budget={sum(budgets)}")

    def one_pass(to_host, tm, tx=texts, bd=budgets, model=None):
        # the CFM start noise is drawn from torch's global generator, which torch seeds at random in every process
        torch.manual_seed(SEED + rank)
        return (model or tts).generate_batch(tx, max_new_tokens=bd, seed=1000 * rank, kv_dtype="bf16", to_host=to_host, timings=tm)

    # ---- 1. warm-up + timed region (device-resident inputs, no kernel timers)
    for i in range(args.warmup):
        tmw = {}
        one_pass(False, tmw)
        log(f"warmup {i}: " + json.dumps({k: (round(v, 1) if isinstance(v, float) else v) for k, v in tmw.items()}))
    launches0 = eng.h.launch_count()
    eng.stats.update(paged_bytes=0.0, paged_launches=0, decode_steps=0, decode_row_steps=0)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    last = {"n": 0}

    def timed_step(tm):
        wavs = one_pass(False, tm)
        last["n"] += 1
        if last["n"] == args.steps:       # only the last step's waveforms outlive their step
            last["wavs"] = wavs

    ms, wall, tms = timed(timed_step, args.steps)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last.pop("wavs"), args.budget_max)
    launches = eng.h.launch_count() - launches0
    stats_timed = dict(eng.stats)
    audio_total = allsum(sum(t["audio_s"] for t in tms))
    value = audio_total / (ms / 1000.0)
    log(f"timed: {ms:.1f} ms for {args.steps} steps -> {value:.1f} audio-s/s")
    stage = {k: sum(t[k] for t in tms) / len(tms) for k in ("t3_ms", "flow_ms", "hift_ms")}

    # ---- 2. e2e: host token ids in, waveforms back in pinned host memory (copies inside the timed region)
    e2e_steps = max(1, min(2, args.steps))
    # allocator warm-up (like the W warm-up steps of the device path): page-lock the output staging size once, so that the timed
    # passes reuse torch's cached pinned block instead of paying cudaHostAlloc for ~0.5 GB inside the timed region
    _warm = torch.empty(int(sum(budgets)) * 960, dtype=torch.float32, pin_memory=True)
    del _warm
    ms_e, wall_e, tms_e = timed(lambda tm: one_pass(True, tm), e2e_steps)
    audio_e = allsum(sum(t["audio_s"] for t in tms_e))
    log(f"e2e: {ms_e:.1f} ms for {e2e_steps} steps")

    # ---- 3. profiling pass (outside the timed region): CUDA events around every launch of every instrumented kernel class
    prof = {}
    if not args.no_profile:
        eng.stats.update(paged_bytes=0.0, paged_launches=0, decode_steps=0, decode_row_steps=0)
        eng.h.set_option("time_kernel", "all")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        one_pass(False, {})
        e1.record(); torch.cuda.synchronize()
        pass_ms = e0.elapsed_time(e1)
        for cls in ("gemm_tc", "wres", "stream", "gemv", "attn_tc", "flash", "paged", "hift_conv"):
            prof[cls] = eng.h.timer_read_class(cls)
            prof[cls]["pass_ms"] = pass_ms
        prof["paged"]["paged_bytes"] = eng.stats["paged_bytes"]
        eng.h.set_option("time_kernel", "none")
        log("profile pass %.0f ms: " % pass_ms + ", ".join(f"{k} {v['ms']:.0f} ms / {v['n']}" for k, v in prof.items()))

    # ---- 4a. strong scaling: 256 utterances TOTAL, LPT-sharded (BASELINE config 3 split over the box)
    extra = {}
    if world > 1 and not args.no_extra:
        gt, gb = make_workload(args.batch, SEED, 0, args.budget_max)           # the same global batch on every rank
        shards = shard_utterances([utterance_cost(int(t.numel()), b) for t, b in zip(gt, gb)], world)
        mine = shards[rank]
        tx, bd = [gt[i] for i in mine], [gb[i] for i in mine]
        one_pass(False, {}, tx, bd)
        ms_s, _, tm_s = timed(lambda tm: one_pass(False, tm, tx, bd), 1)
        a_s = allsum(tm_s[0]["audio_s"])
        my_ms = tm_s[0]["t3_ms"] + tm_s[0]["flow_ms"] + tm_s[0]["hift_ms"]
        extra["strong_256"] = {"utterances_total": args.batch, "sharding": "LPT by cost model (chatterbox_b200.dist.utterance_cost)",
                               "audio_s_per_s": a_s / (ms_s / 1000.0), "ms": ms_s, "rank_ms_max": allmax(my_ms), "rank_ms_min": -allmax(-my_ms),
                               "rank0_stage_ms": {k: tm_s[0][k] for k in ("t3_ms", "flow_ms", "hift_ms")},
                               "limiter": "the per-rank AR decode tail: every rank still runs max(budget) sequential decode steps "
                                          "while its row count (and with it the tensor work per step) falls 1/N"}
        log("strong_256: " + json.dumps(extra["strong_256"]))

    if rank == 0 and world == 1 and not args.no_extra:
        # ---- 4d. BASELINE config 2: one utterance (CFG pair), 150 speech tokens = 6 s of audio: latency / RTF
        g1 = torch.Generator().manual_seed(1234)
        text1 = [torch.randint(1, 255, (100,), generator=g1)]
        one_pass(True, {}, text1, [150])
        tm1 = {}
        one_pass(True, tm1, text1, [150])
        b1_ms = tm1["t3_ms"] + tm1["flow_ms"] + tm1["hift_ms"] + tm1["d2h_ms"]
        extra["b1_latency"] = {"audio_s": tm1["audio_s"], "latency_ms": b1_ms, "rtf": b1_ms / 1000.0 / max(tm1["audio_s"], 1e-9),
                               "t3_ms": tm1["t3_ms"], "flow_ms": tm1["flow_ms"], "hift_ms": tm1["hift_ms"],
                               "t3_ms_per_token": tm1["t3_ms"] / 150.0}
        log("B=1 latency: " + json.dumps(extra["b1_latency"]))

    # ---- 4b / 4c. the other model families need other checkpoints: free this one first
    del tts, t3, s3
    eng._t3_bufs.clear(); eng._ws = None
    del eng
    torch.cuda.empty_cache()

    def family(name, build, vocab_lo, vocab_hi, total, cfg_rows, nfe):
        """One warm + one timed pass of `total` utterances sharded over the ranks (LPT), for another checkpoint."""
        e2 = Engine(local_rank)
        model = build(e2)
        gt, gb = make_workload(total, SEED + 17, 0, args.budget_max, vocab_lo, vocab_hi)
        shards = shard_utterances([utterance_cost(int(t.numel()), b) for t, b in zip(gt, gb)], world)
        tx, bd = [gt[i] for i in shards[rank]], [gb[i] for i in shards[rank]]
        kw = dict(seed=1000 * rank, kv_dtype="bf16", to_host=False)
        run = (lambda tm: model.generate_batch(tx, max_new_tokens=bd, timings=tm, **kw)) if name != "turbo_512" else \
              (lambda tm: model.generate_batch(tx, max_gen_len=bd, timings=tm, **kw))
        run({})
        ms_f, _, tm_f = timed(run, 1)
        a_f = allsum(tm_f[0]["audio_s"])
        out = {"utterances_total": total, "utterances_this_rank": len(tx), "audio_s_per_s": a_f / (ms_f / 1000.0), "ms": ms_f,
               "audio_s": a_f, "rank0_stage_ms": {k: tm_f[0][k] for k in ("t3_ms", "flow_ms", "hift_ms")}}
        model = None
        e2._t3_bufs.clear(); e2._ws = None
        del e2
        torch.cuda.empty_cache()
        log(f"{name}: " + json.dumps(out))
        return out

    if not args.no_extra:
        def build_mtl(e2):      # BASELINE config 4: Chatterbox-Multilingual (text vocabulary 2454, t3_config.py:28-41)
            from chatterbox_b200 import ChatterboxMultilingualTTS
            t = T3(e2, W.make_t3_weights(1, text_vocab=2454))
            s = S3Gen(e2, W.make_flow_weights(0), W.make_hift_weights(0))
            return ChatterboxMultilingualTTS(t, s, None, f"cuda:{local_rank}", Conditionals(T3Cond(**c3), cg))

        def build_turbo(e2):    # BASELINE config 5: Turbo 350M (GPT-2 medium T3, no CFG, 2-step meanflow)
            from chatterbox_b200 import ChatterboxTurboTTS
            t = T3(e2, W.make_t3_turbo_weights(0))
            s = S3Gen(e2, W.make_flow_weights(0, meanflow=True), W.make_hift_weights(0), meanflow=True)
            ct, cgt = W.make_conds(1234, n_t3_prompt=375)
            return ChatterboxTurboTTS(t, s, None, f"cuda:{local_rank}", Conditionals(T3Cond(**ct), cgt))

        extra["mtl_256"] = family("mtl_256", build_mtl, 1, 2454, 256, 2, 10)
        extra["mtl_256"]["note"] = "23-language mixed batch: on the hot path the language only changes token ids ([lang] prefix), ids ~ randint(1, 2454)"
        extra["turbo_512"] = family("turbo_512", build_turbo, 0, 50276, 512, 1, 2)
        extra["turbo_512"]["note"] = "1 T3 row per utterance (no CFG), +3 silence tokens, 2 meanflow NFE, HiFT"

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rooflines
    n_gen = budgets                                     # random weights: utterances run to their budget (EOS is ~1e-4 per step)
    wk = stage_work(texts, n_gen)
    stage_roof = {
        "t3": {"bound": "hbm", "achieved": wk["t3_bytes"] / 1e9 / (stage["t3_ms"] / 1e3), "peak": hbm_peak, "unit": "GB/s",
               "frac": wk["t3_bytes"] / 1e9 / (stage["t3_ms"] / 1e3) / hbm_peak,
               "model": "decode steps x 1.0234 GB of weights + KV read/write (BASELINE.md 4); prefill time included in the stage"},
        "flow": {"bound": "tensor", "achieved": wk["flow_flops"] / 1e12 / (stage["flow_ms"] / 1e3), "peak": tf_peak, "unit": "TFLOP/s",
                 "frac": wk["flow_flops"] / 1e12 / (stage["flow_ms"] / 1e3) / tf_peak,
                 "model": "encoder 113.2 MFLOP*n + 90.1 kFLOP*n^2; CFM T*(132.16 M + 114 688*T) per NFE and row, 2 rows x 10 NFE"},
        "hift": {"bound": "tensor+hbm", "achieved": wk["hift_flops"] / 1e12 / (stage["hift_ms"] / 1e3), "peak": tf_peak, "unit": "TFLOP/s",
                 "frac": wk["hift_flops"] / 1e12 / (stage["hift_ms"] / 1e3) / tf_peak,
                 "hbm_view": {"achieved": wk["hift_bytes"] / 1e9 / (stage["hift_ms"] / 1e3), "peak": hbm_peak, "unit": "GB/s",
                              "frac": wk["hift_bytes"] / 1e9 / (stage["hift_ms"] / 1e3) / hbm_peak,
                              "model": "0.30 MB per mel frame (fused model, SURVEY.md 8d)"},
                 "model": "612.3 MFLOP per mel frame"}}
    traffic = {}
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")      # dram__bytes per launch from the committed ncu --set full captures
    if os.path.exists(tp):
        traffic = json.load(open(tp))
    kroof = {}
    if prof:
        def entry(cls, kernel, what, bound, note=None, bytes_override=None):
            r = prof[cls]
            if r["n"] == 0:
                return
            sec = r["ms"] / 1e3
            byt = bytes_override if bytes_override is not None else r["bytes"]
            e = {"what": what, "bound": bound, "launches": r["n"], "avg_launch_ms": r["ms"] / r["n"], "share_of_step": r["ms"] / r["pass_ms"],
                 "algorithmic_flops_per_launch": r["work"] / r["n"], "algorithmic_bytes_per_launch": byt / r["n"],
                 "tflops": r["work"] / 1e12 / sec if sec > 0 else 0.0, "gbytes_per_s": byt / 1e9 / sec if sec > 0 else 0.0}
            if bound == "hbm":
                e.update(achieved=e["gbytes_per_s"], peak=hbm_peak, unit="GB/s")
            else:
                e.update(achieved=e["tflops"], peak=tf_peak, unit="TFLOP/s")
            e["frac"] = e["achieved"] / e["peak"]
            tr = traffic.get(kernel)
            e["traffic"] = tr["dram_bytes_per_launch"] if tr else None       # dram__bytes_read + write per launch (ncu --set full)
            if tr:
                e["traffic_note"] = f"ncu capture {tr['from']} (profiles/), taken at the capture's own launch shape"
            if note:
                e["note"] = note
            kroof[kernel] = e
        entry("gemm_tc", "gemm_tc_kernel", "tcgen05 GEMM / implicit-GEMM conv, one tile per CTA (CFM convs + ff2, encoder, T3 prefill, HiFT pre/up/post convs)", "tensor",
              "algorithmic flops = 2*M*N*K; bf16 hi/lo operands issue 2x on the tensor pipe")
        entry("wres", "gemm_wres_kernel", "weight-resident persistent GEMM of the CFM block projections (K <= 512), TMA-store epilogue", "hbm",
              "K = 256: 95 FLOP/B, below the ridge (222 FLOP/B): HBM-bound by its activations")
        entry("stream", "gemm_stream_kernel", "persistent GEMM of the T3 decode-step projections (weights streamed once per step)", "hbm")
        entry("gemv", "gemv_kernel", "weight-streaming GEMV (<= 8 rows)", "hbm")
        entry("attn_tc", "attn_otm_kernel", "tcgen05 flash attention of the CFM estimator blocks (fp16 operands, P and O in TMEM)", "tensor",
              "algorithmic flops = 4*64*heads*sum(T^2); head dim 64: 8192 ex2 per 128x64 block = 512 MUFU clocks against 256 MMA clocks -> <= ~50 % of the tensor peak")
        entry("flash", "flash_attn_kernel", "mma.sync flash attention (conformer encoder with rel-pos bias, T3 prefill)", "tensor", "legacy path; time share only")
        entry("paged", "paged_bulk_kernel", "T3 decode attention over the paged KV cache (bulk-copy staged, fused RoPE + append)", "hbm",
              bytes_override=prof["paged"]["paged_bytes"])
        entry("hift_conv", "hift_conv_kernel", "HiFT ResBlock convolutions (persistent, row-shifted UMMA descriptors)", "tensor",
              "algorithmic flops = 2*rows*C*k*C; bf16 hi/lo operands issue 2x")
        dom = max(kroof, key=lambda k: kroof[k]["share_of_step"])
        roofline = dict(kernel=dom, **{k: v for k, v in kroof[dom].items() if k != "what"})
        roofline["measured_in"] = "separate profiling pass after the timed region (CUDA events per launch on the launching stream)"
    else:
        roofline = {"bound": "tensor", "achieved": stage_roof["flow"]["achieved"], "peak": tf_peak, "unit": "TFLOP/s",
                    "frac": stage_roof["flow"]["frac"], "traffic": None, "kernel": "flow stage (profiling passes disabled)"}

    cpu_base = None
    if world == 1 and args.cpu_sample != "none":
        log(f"cpu baseline on {host_threads()} threads (os.cpu_count={os.cpu_count()})")
        cpu_base = cpu_baseline_k4(texts, budgets)
        log(f"cpu baseline done: {cpu_base['wall_s']} s for {cpu_base['audio_s']} s of audio")

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16 weights/KV, fp32 residual stream + accumulate; T3 decode and CFM block operands one fp16 plane, CFM convs / encoder / HiFT operands bf16 hi+lo planes",
        "data": "synthetic",
        "rtf": (ms / 1000.0) / audio_total * world,
        "config": {"workload": WORKLOAD,
                   "utterances_per_gpu": args.batch, "global_batch": args.batch * world, "parallelism": f"utterance-sharded dp{world}",
                   "weights": "seeded random init of the reference architecture (532M T3 + 112M flow + 21M HiFT)",
                   "l2_policy": "working set >> L2 (KV pages ~40 GB, activations GBs); no explicit flush needed",
                   "audio_s_per_step_per_gpu": sum(t["audio_s"] for t in tms) / args.steps, "stage_ms": stage,
                   "decode_steps_per_step": stats_timed["decode_steps"] / args.steps, "peaks": peak_src,
                   "stage_rooflines": stage_roof, "kernel_rooflines": kroof, **extra},
        "clocks": clk,
        "gpu_launches": int(launches),
        "e2e": {"value": audio_e / (ms_e / 1000.0), "unit": UNIT, "steps": e2e_steps,
                "h2d_bytes_per_step": int(tms_e[0]["h2d_bytes"]), "d2h_bytes_per_step": int(tms_e[0]["d2h_bytes"]),
                "wall_s": wall_e},
        "roofline": roofline,
    }
    if cpu_base is not None:
        line["cpu_baseline"] = cpu_base
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("CBX_BENCH_WATCHDOG", 2400)), exit=True, file=sys.stderr)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--budget-max", type=int, default=1000, help="upper bound of the per-utterance token budget (debug)")
    ap.add_argument("--no-profile", action="store_true", help="skip the per-kernel-class profiling passes")
    ap.add_argument("--no-extra", action="store_true", help="skip strong scaling / multilingual / Turbo / B=1 passes")
    ap.add_argument("--cpu-sample", default="k4", choices=["k4", "none"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the waveforms of the last timed step (rank 0) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_engine(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
