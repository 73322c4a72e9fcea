#!/usr/bin/env python
"""bench.py - speech-tokens/s of the GPT decode hot path (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference|torch-cuda]
                    [--config c2|c3] [--path gpt|decoder] [--dump-outputs DIR]

A "step" is one whole ``generate`` pass of the hot path over one batch: a 16-token prompt and
``--tokens`` (512) forced speech tokens per row, greedy + EOS excluded (BASELINE.json configs[1];
SURVEY.md 8d C2).  ``value`` = speech tokens/s with inputs resident in HBM (prompt embeddings,
mask, Exp(1) noise already on the device; CUDA events on the launching stream).  ``e2e`` = the same
metric through the public ``GPT.generate`` call with HOST buffers (pinned prompt embeddings +
noise H2D, sampled ids D2H inside the timed region).  N > 1: one process per GPU (torchrun),
utterances sharded, one NCCL broadcast of the packed weights at load, no step-loop collective.

``--config c3``: BASELINE configs[2] (batch 32, prompts of 8..128 tokens, refine-text pass then code pass, top-p 0.7 /
top-k 20 / penalty 1.05).  ``--path decoder``: hot path 2 at BASELINE configs[3] (DVAE decoder + Vocos + iSTFT of
64 x 10 s), audio-samples/s with a tensor-core roofline against a TF32 peak measured in the same run.
``--impl torch-cuda``: the reference's own stack (HF LlamaModel, torch SDPA, eager PyTorch) on the same B200.
``--dump-outputs DIR``: after the timed steps, what the timed path returned in its last step (rank 0) goes to
``DIR/<name>.npy`` as float32; inputs are seeded, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

PROMPT_LEN = 16
# SURVEY.md 8d: streamed weight elements per audio step (20 layers + 41 norms + 4 heads)
W_ELEMS = 190_698_240
KV_BYTES_PER_TOKEN_ROW = 20 * 2 * 768 * 4  # 122,880 B per row per context token (read), same per step (write)
# dram__bytes_read.sum + dram__bytes_write.sum of ONE single-step k_flow<1> launch (ncu --set full, round 2; see profiles/)
TRAFFIC_K_FLOW_B1 = 771_000_000


def algorithmic_bytes_per_step(B: int, T: float) -> float:
    return W_ELEMS * 4 + B * T * KV_BYTES_PER_TOKEN_ROW + B * KV_BYTES_PER_TOKEN_ROW


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(self.rows[0][1]), "reasons": reasons,
                "samples": len(sm)}


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each array as ``out_dir/<name>.npy`` in float32 (token ids are exact in float32: they are < 2**24)."""
    import numpy as np

    host = {name: a.detach().cpu().numpy().astype(np.float32) for name, a in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"outputs of {total} B exceed the {DUMP_LIMIT_BYTES} B dump limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def build_inputs(B: int, tokens: int, seed: int):
    from chattts_b200.processors import ArgmaxOnly, build_sampler_config, exp_noise, gen_logits
    from chattts_b200.prompts import synth_prompt_batch

    ids, mask, tmask = synth_prompt_batch([PROMPT_LEN] * B, seed=seed)
    warp, proc = gen_logits(num_code=625, top_P=0.7, top_K=20, repetition_penalty=1.05)
    procs = (*proc, *warp, ArgmaxOnly(exclude_eos=True))
    cfg = build_sampler_config(procs, [0.3] * 4, 625, tokens)
    q = exp_noise(B * 4, 626, 1234)
    return ids, mask, tmask, procs, cfg, q


def run_ours(args, rank: int, world: int, local_rank: int):
    import torch.distributed as dist

    from chattts_b200 import _lib
    from chattts_b200.config import Config
    from chattts_b200.dist import broadcast_weights
    from chattts_b200.embed import Embed
    from chattts_b200.gpt import GPT
    from chattts_b200.synth import synth_embed_state, synth_gpt_state

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    cfg = Config()
    B, tokens = args.batch, args.tokens
    es = synth_embed_state(1)
    embed = Embed(768, 626, 21178, 4).load_state_dict(es).to(dev)
    gpt = GPT(cfg.gpt, embed, device=dev, device_gpt=dev, max_batch=max(B, 32), max_context=PROMPT_LEN + tokens + 128)
    if world > 1:
        # one NCCL broadcast of the packed blob at load (SURVEY.md 8e); only rank 0 builds it
        blob = broadcast_weights(gpt, synth_gpt_state(0) if rank == 0 else None, src=0)
        gpt.load_state(None, weights_blob=blob)
    else:
        gpt.load_state(synth_gpt_state(0))

    ids, mask, tmask, procs, scfg, q = build_inputs(B, tokens, seed=1 + rank)
    emb_host = embed(ids, tmask).cpu().pin_memory()
    # ---- resident buffers for `value`
    emb_d, mask_d, q_d = emb_host.to(dev), mask.to(dev).to(torch.uint8), q.to(dev)
    ids_out = torch.zeros(B, tokens, 4, dtype=torch.int32, device=dev)

    def step_resident():
        gpt.enqueue_generate(emb_d, mask_d, scfg, q_d, tokens, False, ids_out, None)

    def step_e2e():
        out = list(gpt.generate(emb_host, ids, temperature=torch.tensor([0.3] * 4), eos_token=625,
                                attention_mask=mask, max_new_token=tokens, min_new_token=tokens,
                                logits_processors=procs, return_hidden=False, show_tqdm=False, manual_seed=1234))[-1]
        return [t.cpu() for t in out.ids]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()
    l0 = lib.ctb_launch_count()
    with ClockSampler(local_rank) as clk:
        ms = timed(step_resident, args.steps)
    launches = int(lib.ctb_launch_count() - l0)
    ms_per_step = ms / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"ids": ids_out})  # [B, tokens, 4] speech-token ids of the last step
    value = world * B * tokens / (ms_per_step / 1e3)

    # ---- e2e through the public API with host buffers
    for _ in range(max(1, min(args.warmup, 2))):
        step_e2e()
    e2e_steps = max(1, min(args.steps, 3))
    ms_e2e = timed(step_e2e, e2e_steps) / e2e_steps
    e2e_value = world * B * tokens / (ms_e2e / 1e3)
    h2d = emb_host.numel() * 4 + mask.numel() + q.numel() * 4
    d2h = B * tokens * 4 * 4 + (16 + 5 * B) * ((tokens + 31) // 32 + 1)

    if rank != 0:
        return None

    # ---- roofline of the dominant kernel, timed live with CUDA events on the launching stream
    peak, peak_src = measured_peaks()
    stream_ptr = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    step_resident()
    torch.cuda.synchronize()

    def time_kind(kind, reps, per_call):
        for _ in range(3):
            _lib.check(lib.ctb_gpt_profile_kernel(gpt._handle, kind, stream_ptr))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            _lib.check(lib.ctb_gpt_profile_kernel(gpt._handle, kind, stream_ptr))
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / (reps * per_call)  # us per launch

    t_avg = PROMPT_LEN + tokens / 2
    step_bytes = algorithmic_bytes_per_step(B, t_avg)
    step_us = ms_per_step * 1e3 / tokens  # `tokens` loop iterations per pass; the 16-token prompt is one batched prefill inside the first
    one_kernel = B <= 4 and not os.environ.get("CTB_NO_FLOW")
    kern = {}
    if one_kernel:
        # B <= 4: the decode loop is the persistent dataflow kernel k_flow (csrc/flow.cuh): one launch = 16 decode
        # iterations (20 layers + heads + sampling tail each).  Timed with CUDA events around single launches.
        roof_new = tokens + 112
        ids_big = torch.zeros(B, roof_new, 4, dtype=torch.int32, device=dev)
        from chattts_b200.processors import build_sampler_config
        scfg_roof = build_sampler_config(procs, [0.3] * 4, 625, roof_new)
        gpt.enqueue_generate(emb_d, mask_d, scfg_roof, q_d, roof_new, False, ids_big, None, n_steps=tokens - 1)
        _lib.check(lib.ctb_gpt_profile_kernel(gpt._handle, 8, stream_ptr))  # warm-up launch (16 steps)
        torch.cuda.synchronize()
        ctx0 = PROMPT_LEN + tokens + 16  # context at the first timed iteration
        reps, per = 5, 16
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            _lib.check(lib.ctb_gpt_profile_kernel(gpt._handle, 8, stream_ptr))
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / reps  # us per launch
        kbytes = sum(algorithmic_bytes_per_step(B, ctx0 + i) for i in range(reps * per)) / reps
        achieved = kbytes / (us * 1e-6) / 1e9
        roofline = {"bound": "hbm", "kernel": f"k_flow<{1 if B == 1 else 2 if B == 2 else 4}> (one launch = {per} decode iterations: "
                                              "20 layers + heads + sampling tail each, no grid barriers)",
                    "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                    "traffic": TRAFFIC_K_FLOW_B1 * per if B == 1 else None, "peak_source": peak_src,
                    "bytes_per_launch": int(kbytes), "us_per_launch": round(us, 2), "steps_per_launch": per,
                    "us_per_step_in_kernel": round(us / per, 2), "context_tokens": [ctx0, ctx0 + reps * per],
                    "traffic_note": "dram__bytes_read+write of one single-step k_flow<1> launch from ncu --set full "
                                    "(profiles/r02_k_flow_b1_full_raw.csv), times the steps per launch; a constant from "
                                    "that capture, not measured in this run"}
    else:
        for kind, name in ((3, "gateup"), (4, "down"), (0, "qkv"), (2, "oproj"), (1, "k_attn"), (5, "heads"), (6, "k_sample")):
            kern[name] = time_kind(kind, 20, 20 if kind < 5 else 1)
        gu_bytes = 2 * 3072 * 768 * 4 + B * 768 * 4 + B * 3072 * 4  # weights + x in + mlp out
        achieved = gu_bytes / (kern["gateup"] * 1e-6) / 1e9
        kname = "k_tc_dec<DE_GATEUP> (tcgen05 3xTF32)" if B > 16 else "k_gemv<BT,EPI_GATEUP>"
        roofline = {"bound": "hbm", "kernel": kname, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                    "frac": round(achieved / peak, 4), "traffic": None, "peak_source": peak_src,
                    "bytes_per_launch": gu_bytes, "us_per_launch": round(kern["gateup"], 3),
                    "kernel_us": {k: round(v, 3) for k, v in kern.items()}}
    roofline["whole_step"] = {"algorithmic_bytes": int(step_bytes), "us": round(step_us, 2),
                              "achieved_gbs": round(step_bytes / (step_us * 1e-6) / 1e9, 1),
                              "frac": round(step_bytes / (step_us * 1e-6) / 1e9 / peak, 4)}

    # ---- the metric at the other batch sizes it is quoted on, and hot path 2 (BASELINE configs[3]); short runs
    sweep = {}
    if world == 1 and not args.no_sweep:
        del gpt
        torch.cuda.empty_cache()
        for bb in (2, 4, 8, 32):
            g2 = GPT(cfg.gpt, embed, device=dev, device_gpt=dev, max_batch=bb, max_context=PROMPT_LEN + tokens + 16)
            g2.load_state(synth_gpt_state(0))
            i2, m2, tm2, _, sc2, q2 = build_inputs(bb, tokens, seed=1)
            e2, mk2, qd2 = embed(i2, tm2).to(dev), m2.to(dev).to(torch.uint8), q2.to(dev)
            o2 = torch.zeros(bb, tokens, 4, dtype=torch.int32, device=dev)
            g2.enqueue_generate(e2, mk2, sc2, qd2, tokens, False, o2, None)  # warm-up (graph capture, clocks)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(2):
                g2.enqueue_generate(e2, mk2, sc2, qd2, tokens, False, o2, None)
            e1.record()
            torch.cuda.synchronize()
            ms2 = e0.elapsed_time(e1) / 2
            sb = algorithmic_bytes_per_step(bb, t_avg)
            us2 = ms2 * 1e3 / tokens
            sweep[f"batch_{bb}"] = {"value": round(bb * tokens / (ms2 / 1e3), 1), "unit": "speech-tokens/s",
                                    "ms_per_step": round(ms2, 2), "rtf": round((ms2 / 1e3) / (bb * tokens * 512 / 24000.0), 6),
                                    "step_us": round(us2, 1), "hbm_frac": round(sb / (us2 * 1e-6) / 1e9 / peak, 4)}
            del g2
            torch.cuda.empty_cache()
        sweep["decoder_c4"] = bench_decoder(dev)

    # the CPU baseline is timed on rank 0 at N = 1 only (it would otherwise compete with the other ranks' host threads)
    cpu = cpu_baseline_sample(B) if world == 1 else None
    audio_s = B * tokens * 512 / 24000.0
    line = {
        "metric": "speech-tokens/sec (GPT decode loop, 4-codebook tokens; RTF = wall / audio seconds @ 24 kHz)",
        "value": round(value, 2), "unit": "speech-tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded random-init weights of the ChatTTS GPT shape)",
        "config": {"workload": f"GPT decode: batch {B}/GPU x (16-token prompt + {tokens} forced speech tokens), greedy "
                               "(BASELINE configs[1]); one step = one whole generate pass",
                   "batch_per_gpu": B, "tokens": tokens, "prompt_len": PROMPT_LEN, "parallelism": f"dp{world}",
                   "l2_policy": "inputs larger than L2: every decode iteration streams 763 MB of fp32 weights (> 126 MB L2)"},
        "rtf": round((ms_per_step / 1e3) / audio_s, 6),
        "e2e": {"value": round(e2e_value, 2), "unit": "speech-tokens/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": round(ms_e2e, 3),
                "rtf": round((ms_e2e / 1e3) / audio_s, 6)},
        "gpu_launches": launches, "clocks": clk.summary(), "roofline": roofline, "cpu_baseline": cpu,
    }
    if sweep:
        line["other_configs"] = sweep
    return line


def bench_decoder(dev, B: int = 64, T: int = 469):
    """Hot path 2 at BASELINE configs[3]: DVAE decoder + Vocos + iSTFT of 10 s of hidden states, batch 64."""
    from chattts_b200.config import Config
    from chattts_b200.decoder import DVAE, Vocos
    from chattts_b200.synth import synth_dvae_state, synth_vocos_state

    cfg = Config()
    voc = Vocos(cfg.vocos, dev, max_batch=B, max_tokens=T)
    voc.state = synth_vocos_state(5)
    dec = DVAE(cfg.decoder, dim=cfg.decoder.idim, device=dev, vocos=voc, max_batch=B, max_tokens=T)
    dec.load_state_dict(synth_dvae_state(2, cfg.decoder, cfg.decoder.idim))
    x = torch.randn(B, T, 768, generator=torch.Generator().manual_seed(1)).to(dev)
    for _ in range(2):
        wav = dec.engine.tokens_to_wav(x, 1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        wav = dec.engine.tokens_to_wav(x, 1)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    frames = B * 2 * T
    flops = frames * 78.7e6  # SURVEY.md 8d: 78.7 MFLOP per mel frame on the hidden path
    return {"workload": f"DVAE decoder + Vocos + iSTFT, batch {B} x {T} tokens (10 s each), hidden path, tcgen05 3xTF32 GEMMs",
            "ms": round(ms, 2), "audio_samples_per_s": round(wav.numel() / (ms / 1e3), 1),
            "rtf": round((ms / 1e3) / (wav.numel() / 24000.0), 7), "tflops_fp32_equiv": round(flops / (ms / 1e3) / 1e12, 1)}


# ------------------------------------------------------------------ hot path 2 as its own benchmark line
DEC_B, DEC_T = 64, 469                      # BASELINE configs[3]: 64 utterances of 10 s (469 tokens = 938 mel frames)
DEC_FLOP_PER_FRAME = 78.7e6                 # SURVEY.md 8d: hidden path, decoder 25.86 + vocos 13.50 + iDFT MMAC per frame
DEC_ALGO_BYTES = 92.2e6 + 157.8e6 + 61.4e6  # hiddens in + fp32 weights + waveform out (SURVEY.md 8d, C4)
# dram__bytes_read + dram__bytes_write summed over the 70 launches of one tokens_to_wav call at C4, from the ncu capture of
# this round (tools/dec_profile.py -> profiles/r02_decoder_c4_dram.csv, _summary.txt); a constant from that capture
DEC_TRAFFIC_C4 = 29_863_704_832


def measured_tf32_peak(dev):
    """cuBLAS TF32 GEMM throughput measured live (torch.matmul fp32 with allow_tf32), best of 5: the denominator of the
    path-2 roofline (MEASURED_PEAKS.json carries bf16 only)."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(2):
            a @ b
        torch.cuda.synchronize()
        best = None
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            torch.cuda.synchronize()
            t = e0.elapsed_time(e1)
            best = t if best is None else min(best, t)
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def decoder_cpu_sample(rows: int = 2):
    """Oracle restatement of DVAE decoder + Vocos + iSTFT (oracle/dvae_oracle.py) on the host cores, `rows` utterances
    of 10 s: the CPU baseline of hot path 2."""
    from chattts_b200.config import Config
    from chattts_b200.synth import synth_dvae_state, synth_vocos_state
    from oracle import dvae_oracle as O

    cfg = Config()
    ds, vs = synth_dvae_state(2, cfg.decoder, cfg.decoder.idim), synth_vocos_state(5)
    x = torch.randn(rows, 768, DEC_T, generator=torch.Generator().manual_seed(1))
    cores = os.cpu_count() or 1
    threads = min(cores, 32)
    torch.set_num_threads(threads)
    O.vocos_decode(O.dvae_decode(x[:1], ds), vs)  # warm-up
    t = time.perf_counter()
    wav = O.vocos_decode(O.dvae_decode(x, ds), vs)
    dt = time.perf_counter() - t
    return {"value": round(wav.numel() / dt, 1), "unit": "audio-samples/s", "cores": threads, "kind": "port",
            "sample": f"oracle/dvae_oracle.py dvae_decode + vocos_decode: {rows} utterances x {DEC_T} tokens (10 s each), "
                      f"{threads} torch threads of a {cores}-core host ({dt:.2f} s)"}, dt


def run_decoder(args, rank: int, world: int, local_rank: int):
    """`--path decoder`: audio-samples/s of DVAE decoder + Vocos + iSTFT at BASELINE configs[3], per GPU 64 x 10 s."""
    import torch.distributed as dist

    from chattts_b200 import _lib
    from chattts_b200.config import Config
    from chattts_b200.decoder import DVAE, Vocos
    from chattts_b200.synth import synth_dvae_state, synth_vocos_state

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    cfg = Config()
    voc = Vocos(cfg.vocos, dev, max_batch=DEC_B, max_tokens=DEC_T)
    voc.state = synth_vocos_state(5)
    dec = DVAE(cfg.decoder, dim=cfg.decoder.idim, device=dev, vocos=voc, max_batch=DEC_B, max_tokens=DEC_T)
    dec.load_state_dict(synth_dvae_state(2, cfg.decoder, cfg.decoder.idim))
    x_host = torch.randn(DEC_B, DEC_T, 768, generator=torch.Generator().manual_seed(1 + rank)).pin_memory()
    x_dev = x_host.to(dev)
    wav_host = torch.empty(DEC_B, 512 * DEC_T - 256, dtype=torch.float32).pin_memory()
    last = {}

    def step_resident():
        last["wav"] = dec.engine.tokens_to_wav(x_dev, 1)

    def step_e2e():
        w = dec.engine.tokens_to_wav(x_host.to(dev, non_blocking=True), 1)
        wav_host.copy_(w, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    for _ in range(args.warmup):
        step_resident()
    l0 = lib.ctb_launch_count()
    with ClockSampler(local_rank) as clk:
        ms = timed(step_resident, args.steps) / args.steps
    launches = int(lib.ctb_launch_count() - l0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"wav": last["wav"]})  # [64, 239872] waveforms, 61.4 MB
    del last["wav"]
    samples = DEC_B * (512 * DEC_T - 256)
    value = world * samples / (ms / 1e3)
    step_e2e()
    ms_e2e = timed(step_e2e, max(1, min(args.steps, 5))) / max(1, min(args.steps, 5))
    if rank != 0:
        return None
    tf32_peak = measured_tf32_peak(dev)
    hbm_peak, hbm_src = measured_peaks()
    flops = DEC_B * 2 * DEC_T * DEC_FLOP_PER_FRAME
    ach = flops / (ms / 1e3) / 1e12
    fma_ms = None
    if not args.no_sweep:  # the fp32-FMA twin of the GEMMs (CTB_DECODER_FMA=1): what "no tensor cores on the conv path" costs
        os.environ["CTB_DECODER_FMA"] = "1"
        try:
            voc2 = Vocos(cfg.vocos, dev, max_batch=DEC_B, max_tokens=DEC_T)
            voc2.state = voc.state
            dec2 = DVAE(cfg.decoder, dim=cfg.decoder.idim, device=dev, vocos=voc2, max_batch=DEC_B, max_tokens=DEC_T)
            dec2.load_state_dict(synth_dvae_state(2, cfg.decoder, cfg.decoder.idim))
            dec2.engine.tokens_to_wav(x_dev, 1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dec2.engine.tokens_to_wav(x_dev, 1)
            e1.record()
            torch.cuda.synchronize()
            fma_ms = e0.elapsed_time(e1)
        finally:
            del os.environ["CTB_DECODER_FMA"]
    cpu, _ = decoder_cpu_sample() if world == 1 else (None, None)
    return {
        "metric": "audio-samples/sec (DVAE decoder + Vocos + iSTFT, hidden-state path, 24 kHz)",
        "value": round(value, 1), "unit": "audio-samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (seeded random-init weights of the ChatTTS decoder / Vocos shapes, N(0,1) hidden states)",
        "config": {"workload": f"hot path 2 at BASELINE configs[3]: batch {DEC_B}/GPU x {DEC_T} tokens (10 s each), GPT hidden "
                               "states -> mel -> waveform; one step = one whole batch", "batch_per_gpu": DEC_B, "tokens": DEC_T,
                   "parallelism": f"dp{world}",
                   "l2_policy": "inputs larger than L2: 92 MB of hidden states in, 61 MB of waveform out and ~2 GB of "
                                "intermediate activations per step (> 126 MB L2)"},
        "rtf": round((ms / 1e3) / (world * samples / 24000.0), 8),
        "e2e": {"value": round(world * samples / (ms_e2e / 1e3), 1), "unit": "audio-samples/s",
                "h2d_bytes_per_step": int(x_host.numel() * 4), "d2h_bytes_per_step": int(wav_host.numel() * 4),
                "ms_per_step": round(ms_e2e, 3)},
        "gpu_launches": launches, "clocks": clk.summary(),
        "roofline": {"bound": "tensor", "kernel": "k_tc_gemm_p<EPI> (persistent tcgen05 3xTF32 conv-as-GEMM, two TMEM accumulators; 47 of the call's 70 launches, 94 % of its time)",
                     "achieved": round(ach, 1), "peak": round(tf32_peak, 1), "unit": "TFLOP/s", "frac": round(ach / tf32_peak, 4),
                     "traffic": DEC_TRAFFIC_C4,
                     "peak_source": "measured in this run: torch.matmul fp32 8192^3 with allow_tf32 (cuBLAS TF32), best of 5",
                     "note": "achieved = ALGORITHMIC fp32 flops (4.73 TFLOP at C4) / step time; the 3xTF32 split issues 3 tensor MACs "
                             "per algorithmic MAC, so the tensor pipes do 3x this figure",
                     "tensor_work_frac": round(3 * ach / tf32_peak, 4),
                     "hbm": {"algorithmic_bytes": int(DEC_ALGO_BYTES), "achieved_gbs": round(DEC_ALGO_BYTES / (ms / 1e3) / 1e9, 1),
                             "dram_traffic_gbs": round(DEC_TRAFFIC_C4 / (ms / 1e3) / 1e9, 1),
                             "traffic_note": "traffic = ncu dram bytes of one call (constant from profiles/r02_decoder_c4_dram.csv), "
                                             "96x the algorithmic bytes: the 4x-wide ConvNeXt intermediates round-trip HBM",
                             "peak_gbs": hbm_peak, "peak_source": hbm_src},
                     "fma_twin_ms": None if fma_ms is None else round(fma_ms, 2)},
        "cpu_baseline": cpu,
    }


def run_reference_decoder(args, rank: int):
    if rank != 0:
        return None
    cpu, _ = decoder_cpu_sample()  # warm
    vals = []
    for _ in range(max(1, args.steps)):
        c, dt = decoder_cpu_sample()
        vals.append((c, dt))
    c, dt = sorted(vals, key=lambda t: t[1])[len(vals) // 2]
    return {"impl": "reference", "metric": "audio-samples/sec (DVAE decoder + Vocos + iSTFT, hidden-state path, 24 kHz)",
            "value": c["value"], "unit": "audio-samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(dt * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": "hot path 2 at BASELINE configs[3]; reference arm times 2 of the 64 utterances"},
            "cpu_baseline": c, "e2e": {"value": c["value"], "unit": "audio-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


# ------------------------------------------------------------------ the reference's own stack on the same GPU
def run_torch_cuda(args, rank: int):
    """`--impl torch-cuda` (BASELINE configs[1] "KV-cache kernel vs torch.sdpa"): HF LlamaModel in fp32 with SDPA attention and
    its DynamicCache on the same B200, heads / temperature / penalty / greedy arg-max as eager torch ops - the reference's
    library path (gpt.py:394-596) without its Python generator overhead.  Same synthetic weights, prompt and token count."""
    if rank != 0:
        return None
    import dataclasses

    from transformers import LlamaConfig, LlamaModel

    from chattts_b200.config import Config
    from chattts_b200.embed import Embed
    from chattts_b200.prompts import synth_prompt_batch
    from chattts_b200.synth import synth_embed_state, synth_gpt_state

    dev = torch.device("cuda", 0)
    c = Config().gpt
    lc = LlamaConfig(hidden_size=c.hidden_size, intermediate_size=c.intermediate_size, num_attention_heads=c.num_attention_heads,
                     num_key_value_heads=c.num_key_value_heads, num_hidden_layers=c.num_hidden_layers,
                     max_position_embeddings=c.max_position_embeddings, rms_norm_eps=c.rms_norm_eps, vocab_size=32,
                     attn_implementation="sdpa")
    model = LlamaModel(lc).eval()
    model.load_state_dict(synth_gpt_state(0), strict=False)
    model = model.to(dev).float()
    es = synth_embed_state(1)
    embed = Embed(768, 626, 21178, 4).load_state_dict(es)
    heads = torch.stack([embed.folded_head(f"head_code.{q}") for q in range(4)]).to(dev)        # [4, 626, 768]
    emb_code = torch.stack([es[f"emb_code.{q}.weight"] for q in range(4)]).to(dev)              # [4, 626, 768]
    B, tokens = args.batch, args.tokens
    ids, mask, tmask = synth_prompt_batch([PROMPT_LEN] * B, seed=1)
    emb0 = embed.to(dev)(ids, tmask).to(dev).float() if hasattr(embed, "to") else None
    penalty = torch.pow(torch.tensor(1.05), torch.arange(17)).to(dev)

    @torch.no_grad()
    def gen(n):
        out = model(inputs_embeds=emb0, use_cache=True)
        past, h = out.past_key_values, out.last_hidden_state[:, -1]
        hist = torch.zeros(B, 4, 0, dtype=torch.long, device=dev)
        for i in range(n):
            logits = torch.einsum("bd,qvd->bqv", h, heads) / 0.3
            if hist.shape[2]:
                cnt = torch.nn.functional.one_hot(hist[:, :, -16:], 626).sum(2)
                a = penalty[cnt]
                logits = torch.where(logits < 0, logits * a, logits / a)
            logits[:, :, 625] = -float("inf")
            idx = logits.argmax(-1)                                   # [B, 4]
            hist = torch.cat([hist, idx[:, :, None]], 2)
            x = emb_code[torch.arange(4, device=dev)[None], idx].sum(1, keepdim=True)   # [B, 1, 768]
            out = model(inputs_embeds=x, past_key_values=past, use_cache=True)
            past, h = out.past_key_values, out.last_hidden_state[:, -1]
        return hist

    n = tokens
    for _ in range(max(1, min(args.warmup, 2))):
        gen(min(n, 32))
    torch.cuda.synchronize()
    steps = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        gen(n)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    value = B * n / (ms / 1e3)
    return {"impl": "torch-cuda", "metric": "speech-tokens/sec (GPT decode loop, 4-codebook tokens; RTF = wall / audio seconds @ 24 kHz)",
            "value": round(value, 2), "unit": "speech-tokens/s", "n_gpus": 1, "steps": steps, "warmup": args.warmup,
            "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (same seeded weights / prompt as the other arms)",
            "config": {"workload": f"HF LlamaModel fp32 + SDPA + DynamicCache, eager PyTorch on the same GPU: batch {B} x (16-token prompt + "
                                   f"{n} greedy speech tokens)", "batch_per_gpu": B, "tokens": n, "prompt_len": PROMPT_LEN},
            "us_per_token_step": round(ms * 1e3 / n, 1), "rtf": round((ms / 1e3) / (B * n * 512 / 24000.0), 6)}


# ------------------------------------------------------------------ BASELINE configs[2]
def run_c3(args, rank: int, world: int, local_rank: int):
    """`--config c3`: batch 32 per GPU, prompt lengths U{8..128} (left padded), refine-text pass (infer_text, temperature 0.7,
    top-p 0.7 / top-k 20, no penalty) then code pass (temperature 0.3, top-p 0.7 / top-k 20 / penalty 1.05, seed 42) through
    the public GPT.generate API with host prompts.  Random weights have no meaningful EOS, so both passes run a FORCED
    length (text 128, code `--tokens`); the metric is speech tokens of the code pass over the time of both passes."""
    import torch.distributed as dist

    from chattts_b200 import _lib
    from chattts_b200.config import Config
    from chattts_b200.dist import broadcast_weights
    from chattts_b200.embed import Embed
    from chattts_b200.gpt import GPT
    from chattts_b200.processors import gen_logits
    from chattts_b200.prompts import synth_prompt_batch
    from chattts_b200.synth import synth_embed_state, synth_gpt_state

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    B, tokens, text_tokens = args.batch if args.batch > 1 else 32, args.tokens, 128
    es = synth_embed_state(1)
    embed = Embed(768, 626, 21178, 4).load_state_dict(es).to(dev)
    gpt = GPT(Config().gpt, embed, device=dev, device_gpt=dev, max_batch=B, max_context=128 + max(tokens, text_tokens) + 16)
    if world > 1:
        gpt.load_state(None, weights_blob=broadcast_weights(gpt, synth_gpt_state(0) if rank == 0 else None, src=0))
    else:
        gpt.load_state(synth_gpt_state(0))
    g = torch.Generator().manual_seed(7 + rank)
    lengths = torch.randint(8, 129, (B,), generator=g).tolist()
    ids, mask, tmask = synth_prompt_batch(lengths, seed=1 + rank)
    warp_t, proc_t = gen_logits(num_code=21178, top_P=0.7, top_K=20, repetition_penalty=1.0)
    warp_c, proc_c = gen_logits(num_code=625, top_P=0.7, top_K=20, repetition_penalty=1.05)

    def pipeline():
        emb = embed(ids, tmask)
        list(gpt.generate(emb, ids, temperature=torch.tensor([0.7]), eos_token=21001, attention_mask=mask,
                          max_new_token=text_tokens, min_new_token=text_tokens, logits_processors=(*proc_t, *warp_t),
                          infer_text=True, show_tqdm=False, manual_seed=42))
        out = list(gpt.generate(emb, ids, temperature=torch.tensor([0.3] * 4), eos_token=625, attention_mask=mask,
                                max_new_token=tokens, min_new_token=tokens, logits_processors=(*proc_c, *warp_c),
                                return_hidden=False, show_tqdm=False, manual_seed=42))[-1]
        return [t.cpu() for t in out.ids]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(1, min(args.warmup, 2))):
        pipeline()
    barrier()
    steps = args.steps
    l0 = lib.ctb_launch_count()
    with ClockSampler(local_rank) as clk:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            code_ids = pipeline()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"ids": torch.stack(code_ids)})  # [B, tokens, 4] code-pass ids of the last step
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    launches = int(lib.ctb_launch_count() - l0) // steps
    if rank != 0:
        return None
    value = world * B * tokens / (ms / 1e3)
    peak, peak_src = measured_peaks()
    code_bytes = algorithmic_bytes_per_step(B, sum(lengths) / B + tokens / 2) * tokens
    text_bytes = (algorithmic_bytes_per_step(B, sum(lengths) / B + text_tokens / 2) + 21178 * 768 * 4 - 4 * 626 * 768 * 4) * text_tokens
    return {
        "metric": "speech-tokens/sec (GPT decode loop, 4-codebook tokens; RTF = wall / audio seconds @ 24 kHz)",
        "value": round(value, 2), "unit": "speech-tokens/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (seeded random-init weights of the ChatTTS GPT shape)",
        "config": {"workload": f"BASELINE configs[2]: batch {B}/GPU, prompts of 8..128 tokens (left padded), refine-text pass "
                               f"({text_tokens} forced text tokens) then code pass ({tokens} forced speech tokens), top-p 0.7 / top-k 20 / "
                               "penalty 1.05, through GPT.generate with host prompts (value IS the end-to-end number)",
                   "batch_per_gpu": B, "tokens": tokens, "text_tokens": text_tokens, "prompt_len": "8..128", "parallelism": f"dp{world}",
                   "l2_policy": "inputs larger than L2: every decode iteration streams >= 763 MB of fp32 weights"},
        "rtf": round((ms / 1e3) / (world * B * tokens * 512 / 24000.0), 6),
        "e2e": {"value": round(value, 2), "unit": "speech-tokens/s", "h2d_bytes_per_step": int(ids.numel() * 8 + mask.numel()),
                "d2h_bytes_per_step": int(B * tokens * 16), "ms_per_step": round(ms, 3)},
        "gpu_launches": launches, "clocks": clk.summary(),
        "roofline": {"bound": "hbm", "kernel": "whole pipeline (tcgen05 decode back end at B = 32, both passes)", "achieved":
                     round((code_bytes + text_bytes) / (ms / 1e3) / 1e9, 1), "peak": peak, "unit": "GB/s",
                     "frac": round((code_bytes + text_bytes) / (ms / 1e3) / 1e9 / peak, 4), "traffic": None, "peak_source": peak_src},
        "cpu_baseline": None,
    }


def best_cpu_threads(run4, candidates=(16, 32, 64, 128)):
    """Pick the torch thread count that makes the oracle port fastest on this host (the reference arm must use the
    host as well as it can; more threads are not always faster for a batch-1 GEMV chain)."""
    cores = os.cpu_count() or 1
    best, best_t = None, None
    for n in candidates:
        if n > cores:
            break
        torch.set_num_threads(n)
        run4()
        t = run4()
        if best_t is None or t < best_t:
            best, best_t = n, t
    if best is None:
        best = cores
    torch.set_num_threads(best)
    return best


def cpu_baseline_sample(B: int, budget_s: float = 8.0):
    """The oracle port (torch fp32 CPU, same ops as the reference's HF path) on this host's cores,
    on a bounded sample of the same workload."""
    from chattts_b200.prompts import synth_prompt_batch
    from chattts_b200.synth import synth_embed_state, synth_gpt_state
    from oracle.gpt_oracle import GPTOracle, SamplerParams

    cores = os.cpu_count() or 1
    orc = GPTOracle(synth_gpt_state(0), synth_embed_state(1))
    ids, mask, tmask = synth_prompt_batch([PROMPT_LEN] * B, seed=1)
    sp = SamplerParams(greedy=True, greedy_exclude_eos=True)

    def run(n):
        t = time.perf_counter()
        orc.generate(orc.embed_prompt(ids, tmask), ids, torch.tensor([0.3] * 4), 625, attention_mask=mask,
                     max_new_token=n, min_new_token=n, sampler=sp, manual_seed=1234)
        return time.perf_counter() - t

    threads = best_cpu_threads(lambda: run(4))
    t4 = run(4)
    n = int(max(8, min(256, budget_s / max(t4 / 4, 1e-3))))
    t = run(n)
    return {"value": round(B * n / t, 2), "unit": "speech-tokens/s", "cores": threads, "kind": "port",
            "sample": f"oracle/gpt_oracle.py generate(): batch {B}, 16-token prompt + {n} tokens, {threads} torch threads "
                      f"on a {cores}-core host ({t:.1f} s)", "ms_per_token_step": round(1e3 * t / n, 2)}


def run_reference(args, rank: int):
    """Reference arm: the reference's CPU implementation of the path (oracle port: torch fp32 CPU),
    each step a bounded sample of the same workload."""
    if rank != 0:
        return None
    from chattts_b200.prompts import synth_prompt_batch
    from chattts_b200.synth import synth_embed_state, synth_gpt_state
    from oracle.gpt_oracle import GPTOracle, SamplerParams

    cores = os.cpu_count() or 1
    B, n = args.batch, args.ref_tokens
    orc = GPTOracle(synth_gpt_state(0), synth_embed_state(1))
    ids, mask, tmask = synth_prompt_batch([PROMPT_LEN] * B, seed=1)
    sp = SamplerParams(greedy=True, greedy_exclude_eos=True)

    def gen(k):
        t = time.perf_counter()
        orc.generate(orc.embed_prompt(ids, tmask), ids, torch.tensor([0.3] * 4), 625, attention_mask=mask,
                     max_new_token=k, min_new_token=k, sampler=sp, manual_seed=1234)
        return time.perf_counter() - t

    threads = best_cpu_threads(lambda: gen(4))

    def step():
        gen(n)

    for _ in range(args.warmup):
        step()
    t = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t) / args.steps
    value = B * n / dt
    sample = (f"oracle port of GPT.generate on CPU: batch {B}, 16-token prompt + {n} tokens per step "
              f"(bounded sample of the {args.tokens}-token workload), {threads} torch threads of {cores} cores")
    return {
        "impl": "reference", "metric": "speech-tokens/sec (GPT decode loop, 4-codebook tokens; RTF = wall / audio seconds @ 24 kHz)",
        "value": round(value, 2), "unit": "speech-tokens/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded random-init weights of the ChatTTS GPT shape)",
        "config": {"workload": f"GPT decode: batch {B} x (16-token prompt + {args.tokens} forced speech tokens), greedy "
                               "(BASELINE configs[1]); reference arm times a bounded sample",
                   "batch_per_gpu": B, "tokens": args.tokens, "prompt_len": PROMPT_LEN},
        "rtf": round(dt / (B * n * 512 / 24000.0), 4),
        "cpu_baseline": {"value": round(value, 2), "unit": "speech-tokens/s", "cores": threads, "kind": "port",
                         "sample": sample},
        "e2e": {"value": round(value, 2), "unit": "speech-tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=int(os.environ.get("CTB_BENCH_BATCH", "1")))
    ap.add_argument("--tokens", type=int, default=512)
    ap.add_argument("--ref-tokens", type=int, default=48)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch-cuda"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3"], help="c2: BASELINE configs[1] (default); c3: configs[2]")
    ap.add_argument("--path", default="gpt", choices=["gpt", "decoder"], help="decoder: hot path 2 at BASELINE configs[3]")
    ap.add_argument("--no-sweep", action="store_true", help="skip the short batch-8/32 and decoder side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the timed path returned in "
                    "its last step as DIR/<name>.npy (float32, seeded inputs: comparable between builds)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        line = run_reference_decoder(args, rank) if args.path == "decoder" else run_reference(args, rank)
        if line is not None:
            print(json.dumps(line), flush=True)
        return
    if args.impl == "torch-cuda":
        line = run_torch_cuda(args, rank)
        if line is not None:
            print(json.dumps(line), flush=True)
        return
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.path == "decoder":
            line = run_decoder(args, rank, world, local_rank)
        elif args.config == "c3":
            line = run_c3(args, rank, world, local_rank)
        else:
            line = run_ours(args, rank, world, local_rank)
        if line is not None:
            print(json.dumps(line), flush=True)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
