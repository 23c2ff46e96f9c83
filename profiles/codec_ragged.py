"""Codec time for utterances of different lengths: one ``decode_code`` call per distinct length (chunks of max_batch,
what the facade did before ``decode_code_ragged``) against ragged calls of up to max_batch utterances.

Full NeuCodec decoder shape, seeded synthetic weights, 3xTF32 (the default precision).  Workloads:
  (a) 64 utterances, lengths drawn from U{50..750} frames (1-15 s each), max_batch 64
  (b) 8 utterances from the same distribution, max_batch 8
  (c) one streaming round at batch 8: 8 windows of 81 frames + 4 tails of 10-60 frames, max_batch 8
Every shape is warmed up; the two strategies alternate inside one run and are timed with CUDA events around the whole
strategy (host work between calls included).  Both must give the same samples within 1e-5.

    python profiles/codec_ragged.py [--reps 7] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from neutts_air_b200 import synthetic
from neutts_air_b200.codec import CodecDecoder, CodecShape

SR = 24_000


def power_limit() -> str:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def by_length(dec, items, cap):
    """one decode_code per distinct length, chunks of at most cap (outputs in input order)"""
    out = [None] * len(items)
    groups = {}
    for i, c in enumerate(items):
        groups.setdefault(len(c), []).append(i)
    for idxs in groups.values():
        for j in range(0, len(idxs), cap):
            grp = idxs[j: j + cap]
            pcm = dec.decode_code(torch.stack([items[i] for i in grp])[:, None, :])
            for r, i in enumerate(grp):
                out[i] = pcm[r, 0]
    return out


def ragged(dec, items, cap):
    out = []
    for j in range(0, len(items), cap):
        grp = items[j: j + cap]
        lens = [len(c) for c in grp]
        out += list(torch.split(dec.decode_code_ragged(torch.cat(grp), lens), [dec.shape.hop * n for n in lens]))
    return out


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    shape = CodecShape()
    dec = CodecDecoder(shape, synthetic.codec_weights(shape, 0), device=dev, max_batch=64, max_frames=750)
    g = torch.Generator().manual_seed(2026)
    codes = lambda n: torch.randint(0, 65536, (n,), generator=g, dtype=torch.int32).to(dev)
    lens_a = torch.randint(50, 751, (64,), generator=g).tolist()
    lens_b = torch.randint(50, 751, (8,), generator=g).tolist()
    lens_c = [81] * 8 + torch.randint(10, 61, (4,), generator=g).tolist()
    work = {"a: 64 utterances U{50..750}": (lens_a, 64), "b: 8 utterances U{50..750}": (lens_b, 8),
            "c: streaming round, 8 windows of 81 + 4 tails": (lens_c, 8)}
    res = {"gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "precision": "3xtf32",
           "shape": "full NeuCodec decoder (hidden 1024, depth 12, n_fft 1920, hop 480), synthetic weights seed 0",
           "reps": args.reps, "workloads": {}}
    for name, (lens, cap) in work.items():
        items = [codes(n) for n in lens]
        timed(lambda: by_length(dec, items, cap))               # warm every shape of both strategies
        _, ref = timed(lambda: by_length(dec, items, cap))
        timed(lambda: ragged(dec, items, cap))
        _, got = timed(lambda: ragged(dec, items, cap))
        err = max(float((a - b).abs().max()) for a, b in zip(ref, got))
        t_old, t_new = [], []
        for _ in range(args.reps):                               # alternate the strategies
            t_old.append(timed(lambda: by_length(dec, items, cap))[0])
            t_new.append(timed(lambda: ragged(dec, items, cap))[0])
        med = lambda t: sorted(t)[len(t) // 2]
        audio_s = sum(lens) * shape.hop / SR
        row = {"lengths": lens, "max_batch": cap, "audio_s": audio_s,
               "calls_by_length": sum((len([n for n in lens if n == L]) + cap - 1) // cap for L in set(lens)),
               "calls_ragged": (len(lens) + cap - 1) // cap,
               "by_length_ms": {"median": med(t_old), "min": min(t_old), "max": max(t_old)},
               "ragged_ms": {"median": med(t_new), "min": min(t_new), "max": max(t_new)},
               "by_length_audio_s_per_s": audio_s / (med(t_old) / 1e3), "ragged_audio_s_per_s": audio_s / (med(t_new) / 1e3),
               "speedup": med(t_old) / med(t_new), "max_abs_diff": err}
        assert err < 1e-5, (name, err)
        res["workloads"][name] = row
        print(f"CODEC-RAGGED {name}: {row['calls_by_length']} calls by length {med(t_old):.1f} ms "
              f"[{min(t_old):.1f}-{max(t_old):.1f}] vs {row['calls_ragged']} ragged {med(t_new):.1f} ms "
              f"[{min(t_new):.1f}-{max(t_new):.1f}] -> x{row['speedup']:.2f}; {row['ragged_audio_s_per_s']:.0f} audio-s/s; "
              f"max |diff| {err:.1e}", flush=True)
    print(f"CODEC-RAGGED on {res['gpu']}, power limit {res['power_limit']}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
