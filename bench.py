#!/usr/bin/env python
"""Headline benchmark: NeuTTS-Air synthetic 500-prefill / 250-decode utterances -> 24 kHz PCM.

    python bench.py --gpus N --steps K --warmup W            # B200 path (this repo)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's PyTorch CPU path
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's PCM (DIR/pcm.npy)

One "step" = one pass of the hot path over one batch of utterances per GPU: prefill(500) ->
250 decode steps (EOS masked until 250, top-k 50 / T=1 sampling on device) -> NeuCodec decode
to 5.0 s of 24 kHz PCM.  Metric (BASELINE.json): audio-seconds per wall-second, whole job.
N = 1: configs[1] (batch 1) + extra lines for batch 8 / 64 (`batches`), configs[2] (mixed-length
batch 64) and configs[4] (Nano-shaped LM, batch-8 streaming, codec every 50 tokens) under
`extra_configs`.  N > 1: configs[3], global batch 64 sharded 64 / N per GPU, waveform all-gather.
`value`: inputs resident in HBM, CUDA events.  `e2e`: the public class (neutts.NeuTTS) with host
buffers.  `roofline`: the decode kernel that dominates the timed region (bytes per launch / event
time).  Prints ONE JSON line on rank 0.  Synthetic data, seeded random weights at the inferred
NeuTTS-Air / NeuCodec shapes (no checkpoints exist offline) -- see DESIGN.md section 5.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PREFILL, DECODE, HOP, SR = 500, 250, 480, 24000
AUDIO_S = DECODE * HOP / SR  # 5.0 s per utterance


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0,
                    help="utterances per GPU per step; default: 1 on one GPU (configs[1]), 64 / N on N GPUs (configs[3])")
    ap.add_argument("--workload", default="fixed", choices=["fixed", "mixed"],
                    help="fixed: every prompt 500 tokens (configs[1]); mixed: prompt lengths U{200..1400}, seeded (configs[2])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the batch 8 / 64 lines reported under 'batches' (N=1 runs only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the PCM of the last timed step to DIR/pcm.npy (float32, one row per utterance) to compare builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------
# synthetic model + workload (identical on every rank and for both arms)
# ----------------------------------------------------------------------------------------------
def synth_prompts(n, vocab, speech_base, seed, mixed=False):
    """SURVEY §8d: 128 uniform text ids + 372 speech ids (dave.pt-shaped reference), P = 500.
    mixed (configs[2]): P_i ~ U{200..1400}, a quarter of it text ids, the rest reference speech ids."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        P = int(torch.randint(200, 1401, (1,), generator=g)) if mixed else PREFILL
        n_text = P // 4 if mixed else PREFILL - 372
        text = torch.randint(0, 151643, (n_text,), generator=g)
        ref = speech_base + torch.randint(0, 65536, (P - n_text,), generator=g)
        out.append(torch.cat((text, ref)).tolist())
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nme, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU path (transformers generate + codec restatement)
# ----------------------------------------------------------------------------------------------
def reference_components(n_decode, threads=None):
    """Times prefill, decode (tok/s) and codec on the host cores with the reference's code path:
    transformers Qwen2ForCausalLM.generate in fp32 (what transformers 4.56.1 loads by default at
    neutts/neutts.py:164) + the fp32 PyTorch NeuCodec decoder restatement (oracle/codec_oracle.py)."""
    from neutts_air_b200 import synthetic
    from neutts_air_b200.codec import CodecShape
    from oracle import codec_oracle as CO
    from oracle import lm_oracle as LO

    if threads:
        torch.set_num_threads(threads)
    cfg = LO.LMConfig()
    w = LO.LMWeights(embed=None)
    sd = {k: v.float() for k, v in synthetic.lm_state_dict(cfg, 0).items()}   # same bf16-valued weights as the GPU arm
    w.embed, w.final_norm, w.lm_head = sd["model.embed_tokens.weight"], sd["model.norm.weight"], sd["model.embed_tokens.weight"]
    for i in range(cfg.num_layers):
        p = f"model.layers.{i}."
        w.layers.append(dict(ln1=sd[p + "input_layernorm.weight"], ln2=sd[p + "post_attention_layernorm.weight"],
                             wq=sd[p + "self_attn.q_proj.weight"], bq=sd[p + "self_attn.q_proj.bias"],
                             wk=sd[p + "self_attn.k_proj.weight"], bk=sd[p + "self_attn.k_proj.bias"],
                             wv=sd[p + "self_attn.v_proj.weight"], bv=sd[p + "self_attn.v_proj.bias"],
                             wo=sd[p + "self_attn.o_proj.weight"], wg=sd[p + "mlp.gate_proj.weight"],
                             wu=sd[p + "mlp.up_proj.weight"], wd=sd[p + "mlp.down_proj.weight"]))
    model = LO.to_hf_model(cfg, w, attn_implementation="sdpa")
    speech_base, eos = 151936, 151670
    prompt = torch.tensor(synth_prompts(1, cfg.vocab_size, speech_base, 1234)[0])[None]
    ccfg = CO.CodecConfig()
    cd = synthetic.codec_weights(CodecShape(), 0)
    cw = CO.CodecWeights(**{k: cd[k] for k in ("project_out_w", "project_out_b", "fc_post_a_w", "fc_post_a_b", "embed_w", "embed_b",
                                               "prior", "blocks", "post", "final_ln_w", "final_ln_b", "head_w", "head_b")})
    codes = torch.randint(0, 65536, (1, 1, DECODE), generator=torch.Generator().manual_seed(7))

    def run(n_new):
        t0 = time.perf_counter()
        with torch.no_grad():
            model.generate(prompt, max_length=2048, eos_token_id=eos, do_sample=True, temperature=1.0, top_k=50, use_cache=True,
                           min_new_tokens=n_new, max_new_tokens=n_new, pad_token_id=eos)
        return time.perf_counter() - t0

    return dict(run=run, codec=lambda: _timeit(lambda: CO.decode_code(codes, cw, ccfg)), cfg=cfg)


def _timeit(fn):
    t0 = time.perf_counter()
    with torch.no_grad():
        fn()
    return time.perf_counter() - t0


def reference_measure(steps, warmup):
    """Returns (audio-s/s, ms per utterance, sample description, cores)."""
    cores = os.cpu_count() or 1
    comp = reference_components(DECODE)
    comp["run"](1)                           # warm-up (allocator, thread pools)
    # Thread count: the decode loop is a chain of small GEMVs and gets slower with too many threads (460 ms/token
    # at 64 threads on the 128-core GPU box against 64 ms/token at 8), prefill wants many.  Give the reference its
    # best setting: estimate the full workload at a few thread counts from prefill + 8 decode tokens each.
    default_threads = torch.get_num_threads()
    best = None
    for th in sorted({t for t in (4, 8, 16, 32, 64, default_threads) if t <= max(cores, 1)}):
        torch.set_num_threads(th)
        a = comp["run"](1)
        b = comp["run"](9)
        est = a + max((b - a) / 8, 1e-4) * (DECODE - 1)
        if best is None or est < best[0]:
            best = (est, th)
    torch.set_num_threads(best[1])
    t1 = comp["run"](1)                      # prefill-dominated time
    t_short = comp["run"](17)
    per_tok = max((t_short - t1) / 16, 1e-4)
    est_full = t1 + per_tok * (DECODE - 1)
    t_codec = comp["codec"]()
    t_codec = comp["codec"]()
    if est_full * (steps + warmup) <= 240:   # the whole arm stays within a few minutes: run the real workload
        for _ in range(warmup):
            comp["run"](DECODE)
        ts = [comp["run"](DECODE) + comp["codec"]() for _ in range(steps)]
        t = float(np.mean(ts))
        sample = f"full workload x{steps}: generate(500->750, fp32, sdpa) + codec restatement(250 frames), {torch.get_num_threads()} threads"
    else:
        t = est_full + t_codec
        sample = (f"bounded sample: prefill(500)+1 tok = {t1:.2f}s, 16 decode tokens -> {per_tok * 1e3:.1f} ms/token, codec(250) = "
                  f"{t_codec:.2f}s; composed to 250 tokens, {torch.get_num_threads()} threads")
    par = [ln.strip() for ln in torch.__config__.parallel_info().splitlines() if "threads" in ln.lower() or "openmp" in ln.lower()]
    return AUDIO_S / t, t * 1e3, sample, cores, dict(prefill_s=t1, ms_per_token=per_tok * 1e3, codec_s=t_codec,
                                                      decode_tok_s=1.0 / per_tok, torch_threads=torch.get_num_threads(),
                                                      parallel_info="; ".join(par[:4]))


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    v, ms, sample, cores, parts = reference_measure(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "audio-sec/sec (RTF), NeuTTS-Air 500 prefill / 250 decode + NeuCodec decode", "value": v,
        "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: 1 utterance, 500 prefill / 250 decode tokens, batch=1, NeuCodec decode to 24 kHz",
                   "note": "reference never batches (neutts/neutts.py:335); CPU path = transformers generate fp32 + codec restatement"},
        "cpu_baseline": {"value": v, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": sample, **parts},
        "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------
_WEIGHTS = {}
SPEECH_BASE, EOS = 151936, 151670
# dram__bytes_read.sum + dram__bytes_write.sum of ONE decode_tc_kernel launch (249 steps, batch 1, contexts 500..749)
# from profiles/decode_tc_b1_r2_ncu_summary.txt (ncu --set full); None until a capture of the current kernel exists
NCU_TRAFFIC_B1 = 278.50e9


def build_engines(device, batch, prefill_tokens=None):
    from neutts_air_b200 import synthetic
    from neutts_air_b200.codec import CodecDecoder, CodecShape
    from neutts_air_b200.lm import LMShape, SpeechLM

    shape = LMShape()
    if not _WEIGHTS:   # seeded random weights are generated once per process and shared by the sweep engines
        _WEIGHTS["lm"] = synthetic.lm_state_dict(shape, 0)
        _WEIGHTS["codec"] = synthetic.codec_weights(CodecShape(), 0)
    lm = SpeechLM(shape, _WEIGHTS["lm"], device=device, max_batch=batch, max_ctx=2048, max_new=256,
                  max_prefill_tokens=prefill_tokens or batch * PREFILL)
    codec = CodecDecoder(CodecShape(), _WEIGHTS["codec"], device=device, max_batch=batch, max_frames=256)
    return lm, codec


class _BenchTokenizer:
    """The two lookups the facade's hot path makes (neutts/neutts.py: _tok_id / speech_base)."""

    def convert_tokens_to_ids(self, name: str) -> int:
        if name == "<|SPEECH_GENERATION_END|>":
            return EOS
        if name.startswith("<|speech_"):
            return SPEECH_BASE + int(name[9:-2])
        raise KeyError(name)


def make_facade(lm, codec, batch, seed):
    """The public class (neutts.NeuTTS) around the two engines.  One bench-only shim: a random-weight LM emits
    arbitrary vocabulary ids, so the id -> code map folds them into the codebook instead of dropping non-speech ids
    (every utterance then has exactly 250 frames, as a trained model would produce for the workload)."""
    import warnings

    from neutts import NeuTTS

    class BenchTTS(NeuTTS):
        def _ids_to_codes(self, ids):
            return (ids.long() - SPEECH_BASE) % 65536

        def _ids_to_codes_masked(self, ids):
            return (ids.long() - SPEECH_BASE) % 65536, torch.ones_like(ids, dtype=torch.bool)

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return BenchTTS(backbone=lm, codec=codec, tokenizer=_BenchTokenizer(), phonemizer=object(), max_batch=batch, seed=seed)


def step_bytes(shape, B, mean_prompt):
    """Algorithmic HBM bytes of ONE decode step (BASELINE.md §2 / DESIGN.md §4): every bf16 weight once + the KV
    cache of B sequences at the mean context of the 250-token run + the token's activations."""
    p_blk = shape.num_layers * ((shape.num_heads + 2 * shape.num_kv_heads) * 64 * (shape.hidden_size + 1) + shape.hidden_size * shape.num_heads * 64
                                + 3 * shape.hidden_size * shape.intermediate_size + 2 * shape.hidden_size) + shape.hidden_size
    return 2 * (p_blk + shape.vocab_size * shape.hidden_size) + B * (12288 * (mean_prompt + DECODE / 2 + 1) + 2 * shape.hidden_size)


def decode_roofline(lm, B, lens, t_dec, n_steps, launches_per_step):
    """roofline block for the decode loop, the dominant kernel of the timed region."""
    peak, how = peaks()
    sb = step_bytes(lm.shape, B, sum(lens) / len(lens))
    persistent = launches_per_step is None
    alg = sb * n_steps if persistent else sb
    t = t_dec if persistent else t_dec / n_steps
    return {"bound": "hbm",
            "kernel": ("decode_tc_kernel (persistent: all layers + lm_head + sampler, %d decode steps per launch)" % n_steps) if persistent
            else "decode step = CUDA graph of %d kernels (tcgen05 GEMMs, attention, norms, sampler)" % launches_per_step,
            "achieved": alg / t / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / t / 1e9 / peak,
            "traffic": NCU_TRAFFIC_B1 if (persistent and B == 1) else None,
            "traffic_source": "profiles/decode_tc_b1_r2_ncu_summary.txt (dram__bytes_read.sum + dram__bytes_write.sum, one launch)",
            "peak_source": how, "algorithmic_bytes_per_launch": alg, "us_per_launch": t * 1e6,
            "us_per_decode_step": t_dec / n_steps * 1e6, "algorithmic_bytes_per_step": sb}


DUMP_BYTES = 64_000_000


def dump_outputs(path, pcm):
    """PCM of one timed step ([utterances, samples] after the all-gather) -> path/pcm.npy as float32.  The inputs of a
    step depend only on the arguments (seeded prompts, weights and sampling), so two builds can be compared file for
    file.  Beyond DUMP_BYTES a fixed, seeded sample of utterances is written, their indices in path/pcm_rows.npy."""
    os.makedirs(path, exist_ok=True)
    x = pcm.reshape(-1, pcm.shape[-1]).float().cpu().numpy()
    keep = (DUMP_BYTES - 256 - 8 * x.shape[0]) // x[0].nbytes     # 256: the two .npy headers
    if x.shape[0] > keep:
        rows = np.sort(np.random.default_rng(0).choice(x.shape[0], keep, replace=False))
        np.save(os.path.join(path, "pcm_rows.npy"), rows.astype(np.float64))
        x = x[rows]
    np.save(os.path.join(path, "pcm.npy"), x)


def time_decode(lm, prompts, seed=5):
    """(seconds, kernel launches) of the 249-step decode loop alone, CUDA events on the launching stream."""
    sp = lm.sampling(EOS, min_new_tokens=DECODE, max_new_tokens=DECODE, seed=seed)
    lm.prefill(prompts, sp)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = lm.L.nt_launch_count()
    e0.record()
    lm.decode(DECODE - 1, sp)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3, lm.L.nt_launch_count() - n0


def quick_batch(dev, B, steps=2, mixed=False, L=None):
    """One extra line of the metric at another batch size / workload on this GPU (the metric is quoted at batch 1, 8
    and 64; configs[2] is the mixed-length batch 64): inputs resident in HBM, CUDA-event timing, 1 warm-up + `steps`
    timed passes, plus the decode loop alone."""
    prompts = synth_prompts(B, 217472, SPEECH_BASE, 4321, mixed)
    lm, codec = build_engines(dev, B, sum(len(p) for p in prompts))

    def step(seed):
        sp = lm.sampling(EOS, min_new_tokens=DECODE, max_new_tokens=DECODE, top_k=50, temperature=1.0, seed=seed)
        lm.prefill(prompts, sp)
        lm.decode(DECODE - 1, sp)
        c = ((lm.out_tokens[:B, :DECODE].long() - SPEECH_BASE) % 65536)[:, None, :]
        return codec.decode_code(c)

    step(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = L.nt_launch_count() if L else 0
    e0.record()
    for i in range(steps):
        step(10 + i)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / 1e3 / steps
    n1 = L.nt_launch_count() if L else 0
    t_dec, dec_launches = time_decode(lm, prompts)
    lens = [len(p) for p in prompts]
    per_step = None if dec_launches <= 2 else max(1, round(dec_launches / (DECODE - 1)))   # persistent kernel: one launch
    out = {"per_gpu_batch": B, "workload": ("configs[2]: mixed-length prompts U{200..1400} (mean %.0f)" % (sum(lens) / B)) if mixed else "configs[1] shape, 500-token prompts",
           "value": AUDIO_S * B / t, "unit": "audio-s/s", "ms_per_step": t * 1e3, "steps": steps,
           "decode_tok_s": B * (DECODE - 1) / t_dec, "decode_ms_per_token_step": t_dec / (DECODE - 1) * 1e3,
           "gpu_launches_per_pass": int((n1 - n0) / steps) if L else None,
           "roofline": decode_roofline(lm, B, lens, t_dec, DECODE - 1, per_step)}
    del lm, codec
    torch.cuda.empty_cache()
    return out


def stream_line(dev, B=8, frames_per_chunk=50, L=None):
    """configs[4]: NeuTTS-Nano-shaped LM, batch-8 STREAMING synthesis through neutts.NeuTTS (infer_stream_batch's
    engine loop), the codec invoked every 50 generated tokens on the reference's window geometry (lookback 50,
    lookahead 5, overlap 1).  Nano's architecture is not published offline (SURVEY.md §8): the shape is inferred from
    the README's ~229 M total / ~120 M active parameters (hidden 512 from the embedding share)."""
    from neutts_air_b200 import synthetic
    from neutts_air_b200.codec import CodecDecoder, CodecShape
    from neutts_air_b200.lm import LMShape, SpeechLM

    shape = LMShape(vocab_size=217472, hidden_size=512, intermediate_size=2048, num_layers=28, num_heads=8, num_kv_heads=2)
    lm = SpeechLM(shape, synthetic.lm_state_dict(shape, 1), device=dev, max_batch=B, max_ctx=2048, max_new=256, max_prefill_tokens=B * PREFILL)
    if "codec" not in _WEIGHTS:
        _WEIGHTS["codec"] = synthetic.codec_weights(CodecShape(), 0)
    codec = CodecDecoder(CodecShape(), _WEIGHTS["codec"], device=dev, max_batch=B, max_frames=256)
    tts = make_facade(lm, codec, B, seed=99)
    tts.streaming_frames_per_chunk = frames_per_chunk
    tts.streaming_stride_samples = frames_per_chunk * HOP
    prompts = synth_prompts(B, 217472, SPEECH_BASE, 777)
    refs = [[t - SPEECH_BASE for t in p[PREFILL - 372:]] for p in prompts]      # the reference-voice codes inside the prompt

    def run():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        first, samples, rounds = None, 0, 0
        for out in tts._stream_batch(prompts, refs):
            rounds += 1
            n = sum(len(o) for o in out if o is not None)
            if n and first is None:
                first = time.perf_counter() - t0
            samples += n
        return time.perf_counter() - t0, first, samples, rounds

    run()
    n0 = L.nt_launch_count() if L else 0
    t, first, samples, rounds = run()
    launches = (L.nt_launch_count() - n0) if L else None
    ngen = int(lm.n_generated[:B].sum())
    del lm, codec, tts
    torch.cuda.empty_cache()
    return {"workload": f"configs[4]: NeuTTS-Nano-like LM (hidden 512, 28 layers, 8/2 heads, inter 2048; inferred), batch={B} streaming, "
                        f"500-token prompts, codec every {frames_per_chunk} tokens (window {frames_per_chunk}+50+5+1 frames)",
            "per_gpu_batch": B, "value": samples / SR / t, "unit": "audio-s/s", "ms_total": t * 1e3, "first_chunk_ms": first * 1e3 if first else None,
            "audio_s": samples / SR, "generated_tokens": ngen, "decode_tok_s": ngen / t, "rounds": rounds, "gpu_launches": launches,
            "api": "neutts.NeuTTS._stream_batch (engine loop of infer_stream_batch)"}


def main_b200(args):
    import torch.distributed as td

    from neutts_air_b200 import _lib, dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout at the first collective; the contract is ONE JSON line there
        sys.stdout.flush()
        keep = os.dup(1)
        os.dup2(2, 1)
        try:
            td.init_process_group("nccl", device_id=dev)
            td.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(keep, 1)
            os.close(keep)
    L = _lib.lib()
    # N = 1: configs[1] (batch 1, the configuration the metric is quoted on).  N > 1: configs[3], global batch 64
    # sharded 64 / N utterances per GPU (strong scaling: the job is fixed, the GPUs split it).
    B = args.batch if args.batch else (1 if world == 1 else max(1, 64 // world))
    strong = world > 1 and not args.batch
    mixed = args.workload == "mixed"
    prompts = synth_prompts(B, 217472, SPEECH_BASE, 1234 + rank, mixed)
    lens = [len(p) for p in prompts]
    lm, codec = build_engines(dev, B, sum(lens))
    tts = make_facade(lm, codec, B, seed=777)
    h2d_bytes = sum(lens) * 4
    d2h_bytes = B * DECODE * HOP * 4 + B * 256 * 4 + B * 4      # PCM + generated ids + counters read by generate_batch

    def codes_from(lm_):
        return ((lm_.out_tokens[:B, :DECODE].long() - SPEECH_BASE) % 65536)[:, None, :]

    def step_device(seed):
        """inputs already resident in HBM; returns PCM on device."""
        sp = lm.sampling(EOS, min_new_tokens=DECODE, max_new_tokens=DECODE, top_k=50, temperature=1.0, seed=seed)
        lm.prefill(prompts, sp)
        lm.decode(DECODE - 1, sp)
        return codec.decode_code(codes_from(lm))

    def gather(pcm):
        if world > 1:   # the one collective of the path: all-gather of finished waveforms (SURVEY §8e)
            out = torch.empty(world * pcm.shape[0], pcm.shape[2], device=dev)
            td.all_gather_into_tensor(out, pcm[:, 0, :].contiguous())
            return out
        return pcm

    def step_e2e(seed):
        """The call a user makes, minus the text front-end: host prompt ids -> neutts.NeuTTS.infer_from_prompt_ids
        (pinned H2D of the ids, device-side generation, codec, D2H of the PCM) -> host waveforms, then the waveform
        all-gather of the sharded job."""
        tts.seed = seed
        wavs = tts.infer_from_prompt_ids(prompts, max_new_tokens=DECODE, min_new_tokens=DECODE)
        if world > 1:
            mine = list(range(rank * B, rank * B + B))
            wavs = dist.all_gather_waveforms(wavs, mine, world * B, device=dev, t_max=DECODE * HOP)
        assert all(len(w) == DECODE * HOP for w in wavs)
        return wavs

    def barrier():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        gather(step_device(i))
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    n0 = L.nt_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps):
        pcm = gather(step_device(100 + i))
    ev1.record()
    barrier()
    t_dev = ev0.elapsed_time(ev1) / 1e3
    launches = L.nt_launch_count() - n0
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pcm)

    # the parts, each timed alone with CUDA events
    t_dec, dec_launches = time_decode(lm, prompts)
    sp = lm.sampling(EOS, min_new_tokens=DECODE, max_new_tokens=DECODE, seed=5)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    lm.prefill(prompts, sp)
    e1.record()
    torch.cuda.synchronize()
    t_pre = e0.elapsed_time(e1) / 1e3
    e0.record()
    codec.decode_code(codes_from(lm))
    e1.record()
    torch.cuda.synchronize()
    t_codec = e0.elapsed_time(e1) / 1e3

    # end-to-end through the public API and host buffers
    for i in range(2):
        step_e2e(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_e2e(200 + i)
    barrier()
    t_e2e = time.perf_counter() - t0

    times = torch.tensor([t_dev, t_e2e, t_dec, t_pre, t_codec], device=dev, dtype=torch.float64)
    if world > 1:
        td.all_reduce(times, op=td.ReduceOp.MAX)
    t_dev, t_e2e, t_dec, t_pre, t_codec = times.tolist()
    if rank != 0:
        if world > 1:
            td.destroy_process_group()
        return
    total_audio = AUDIO_S * B * world * args.steps
    per_step = None if dec_launches <= 2 else max(1, round(dec_launches / (DECODE - 1)))   # persistent kernel: one launch
    roof = decode_roofline(lm, B, lens, t_dec, DECODE - 1, per_step)
    roof["share_of_timed_region"] = t_dec / (t_dev / args.steps)
    line = {
        "metric": "audio-sec/sec (RTF), NeuTTS-Air 500 prefill / 250 decode + NeuCodec decode",
        "value": total_audio / t_dev, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "bf16 weights+KV / f32 accumulate (LM), 3xTF32 = fp32-grade tensor-core GEMMs (codec)", "data": "synthetic",
        "config": {"workload": (f"configs[2]: mixed-length prompts U{{200..1400}} (mean {sum(lens) / len(lens):.0f}) / 250 decode tokens + NeuCodec "
                                f"decode to 24 kHz, batch={B} per GPU" if mixed else
                                (f"configs[3]: global batch {B * world} sharded {B} utterances/GPU over {world} GPUs, 500 prefill / 250 decode tokens + "
                                 "NeuCodec decode to 24 kHz, NCCL waveform all-gather" if strong else
                                 f"configs[1]: 500 prefill / 250 decode tokens + NeuCodec decode to 24 kHz, batch={B} per GPU")),
                   "per_gpu_batch": B, "global_batch": B * world, "sharding": "utterances one-per-GPU-slot, weights replicated, "
                   "one all-gather of waveforms" if world > 1 else "single GPU",
                   "l2": "inputs larger than L2: 1.1 GB of weights stream per decode step (L2 = 126 MB)", "weights": "seeded random, inferred Air/NeuCodec shapes"},
        "decode_tok_s": B * world * (DECODE - 1) / t_dec,
        "roofline": roof,
        "breakdown_ms": {"prefill": t_pre * 1e3, "decode_249_steps": t_dec * 1e3, "codec": t_codec * 1e3},
        "e2e": {"value": total_audio / t_e2e, "unit": "audio-s/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": t_e2e / args.steps * 1e3, "api": "neutts.NeuTTS.infer_from_prompt_ids" + (" + dist.all_gather_waveforms" if world > 1 else "")},
        "gpu_launches": int(launches),
        "clocks": clk,
    }
    if world == 1 and not args.no_sweep:
        del lm, codec, tts
        torch.cuda.empty_cache()
        line["batches"] = [quick_batch(dev, b, L=L) for b in (8, 64) if b != B]
        line["extra_configs"] = [quick_batch(dev, 64, mixed=True, L=L), stream_line(dev, 8, 50, L=L)]
    if not args.no_cpu_baseline and world == 1:
        try:
            v, ms, sample, cores, parts = reference_measure(1, 0)
            line["cpu_baseline"] = {"value": v, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": sample, **parts}
        except Exception as e:  # the baseline must never take the GPU number down with it
            line["cpu_baseline"] = {"value": None, "unit": "audio-s/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line))
    if world > 1:
        td.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        main_reference(a)
    else:
        main_b200(a)
