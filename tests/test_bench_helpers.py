"""CPU: the measurement harness's own arithmetic (bench.py) -- workload shape, algorithmic bytes of a decode step,
the tokenizer stub the end-to-end leg gives the facade, CLI defaults the driver relies on."""
import os
import sys

import numpy as np
import pytest
import torch

import bench
from neutts_air_b200.lm import LMShape


def test_workload_and_algorithmic_bytes():
    assert (bench.PREFILL, bench.DECODE, bench.HOP, bench.SR) == (500, 250, 480, 24000) and bench.AUDIO_S == 5.0
    p = bench.synth_prompts(3, 217472, bench.SPEECH_BASE, 1)
    assert all(len(x) == 500 for x in p)
    assert all(t < 151643 for t in p[0][:128]) and all(bench.SPEECH_BASE <= t < bench.SPEECH_BASE + 65536 for t in p[0][128:])
    m = bench.synth_prompts(16, 217472, bench.SPEECH_BASE, 2, mixed=True)
    assert all(200 <= len(x) <= 1400 for x in m) and len({len(x) for x in m}) > 4
    # BASELINE.md section 2: every bf16 weight once + KV of the mean context + the token's activations
    sb = bench.step_bytes(LMShape(), 1, 500)
    assert abs(sb - 1.1132e9) < 2e6, sb
    assert abs((bench.step_bytes(LMShape(), 64, 500) - sb) - 63 * (12288 * 626 + 1792)) < 1e3


def test_bench_tokenizer_and_cli_defaults(monkeypatch):
    tok = bench._BenchTokenizer()
    assert tok.convert_tokens_to_ids("<|SPEECH_GENERATION_END|>") == bench.EOS
    assert tok.convert_tokens_to_ids("<|speech_0|>") == bench.SPEECH_BASE
    assert tok.convert_tokens_to_ids("<|speech_65535|>") == bench.SPEECH_BASE + 65535
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    a = bench.parse()
    assert (a.gpus, a.impl, a.batch) == (1, "b200", 0) and a.warmup >= 3 and a.steps >= 1     # contract: W >= 3, default N = 1
    assert a.dump_outputs is None
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "7", "--dump-outputs", "out"])
    a = bench.parse()
    assert (a.steps, a.dump_outputs) == (7, "out")
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse()


def test_dump_outputs_writes_float32_pcm_within_the_budget(tmp_path, monkeypatch):
    pcm = torch.randn(5, 1, 1000)
    bench.dump_outputs(str(tmp_path / "a"), pcm)
    assert sorted(os.listdir(tmp_path / "a")) == ["pcm.npy"]
    got = np.load(tmp_path / "a" / "pcm.npy")
    assert got.dtype == np.float32 and np.array_equal(got, pcm[:, 0].numpy())
    # over the budget: the same seeded subset of utterances every time, indices stored beside it
    monkeypatch.setattr(bench, "DUMP_BYTES", 3 * 4000 + 40 + 256)
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), pcm)
    rows = np.load(tmp_path / "b" / "pcm_rows.npy")
    assert rows.dtype == np.float64 and len(rows) == 3 and np.array_equal(rows, np.load(tmp_path / "c" / "pcm_rows.npy"))
    assert np.array_equal(np.load(tmp_path / "b" / "pcm.npy"), pcm[rows.astype(int), 0].numpy())
    assert sum(f.stat().st_size for f in (tmp_path / "b").iterdir()) <= bench.DUMP_BYTES
