"""CPU: how the facade packs utterances of different lengths into codec calls.  A codec with ``decode_code_ragged``
gets up to ``max_batch`` utterances per call in input order (batch and streaming paths); a codec without it keeps
one ``decode_code`` call per distinct length."""
import numpy as np
import pytest
import torch

from oracle import stream_oracle as SO
from tests.test_host_logic import FakeBatchStreamLM, RampCodec, _tts

HOP = 8


def _ramp(codes: torch.Tensor) -> torch.Tensor:
    """frame i of an item -> HOP samples of code/1000 + 0.01 * i (a misplaced or reordered item changes the output)"""
    c = codes.float()
    return (c[:, None] / 1000.0 + 0.01 * torch.arange(len(c))[:, None] + torch.zeros(1, HOP)).reshape(-1)


class RaggedCodec:
    device = torch.device("cpu")
    hop = HOP

    def __init__(self, max_batch):
        self.max_batch = max_batch
        self.calls = []

    def decode_code(self, codes):
        raise AssertionError("a codec with decode_code_ragged must not get decode_code calls")

    def decode_code_ragged(self, codes, lengths):
        lengths = list(lengths)
        assert codes.dim() == 1 and codes.shape[0] == sum(lengths)
        assert 1 <= len(lengths) <= self.max_batch and min(lengths) >= 1
        self.calls.append(lengths)
        return torch.cat([_ramp(x) for x in torch.split(codes, lengths)])


class GroupingCodec:
    device = torch.device("cpu")

    def __init__(self, max_batch):
        self.max_batch = max_batch
        self.calls = []

    def decode_code(self, codes):
        assert codes.dim() == 3 and codes.shape[1] == 1 and codes.shape[0] <= self.max_batch
        self.calls.append((codes.shape[0], codes.shape[2]))
        return torch.stack([_ramp(codes[r, 0]) for r in range(codes.shape[0])])[:, None, :]


def _utterances(lengths, seed=0):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 65536, (n,), generator=g) for n in lengths]


@pytest.mark.parametrize("max_batch", [1, 3, 4, 16])
def test_ragged_codec_gets_input_order_chunks(max_batch):
    tts, _ = _tts()
    tts.codec = RaggedCodec(max_batch)
    lengths = [7, 1, 30, 7, 12, 2, 30, 5, 9]
    codes = _utterances(lengths)
    wavs = tts._decode_codes(codes)
    want_calls = [lengths[j: j + max_batch] for j in range(0, len(lengths), max_batch)]
    assert tts.codec.calls == want_calls
    assert len(wavs) == len(codes)
    for c, w in zip(codes, wavs):                   # every waveform belongs to its own utterance
        assert isinstance(w, np.ndarray) and w.shape == (HOP * len(c),)
        np.testing.assert_array_equal(w, _ramp(c).numpy())


def test_codec_without_ragged_method_keeps_per_length_grouping():
    tts, _ = _tts()
    tts.codec = GroupingCodec(max_batch=2)
    lengths = [7, 1, 30, 7, 12, 7, 30]
    codes = _utterances(lengths, seed=1)
    wavs = tts._decode_codes(codes)
    assert tts.codec.calls == [(2, 7), (1, 7), (1, 1), (2, 30), (1, 12)]
    for c, w in zip(codes, wavs):
        np.testing.assert_array_equal(w, _ramp(c).numpy())


def test_ragged_rejects_empty_utterance_before_any_call():
    tts, _ = _tts()
    tts.codec = RaggedCodec(4)
    with pytest.raises(ValueError):
        tts._decode_codes(_utterances([3, 0, 2]))
    assert tts.codec.calls == []


class RaggedRampCodec(RampCodec):
    """RampCodec with the ragged entry: records every call's window lengths."""
    max_batch = 2

    def __init__(self):
        self.calls = []

    def decode_code(self, codes):
        raise AssertionError("a codec with decode_code_ragged must not get decode_code calls")

    def decode_code_ragged(self, codes, lengths):
        lengths = list(lengths)
        assert codes.shape == (sum(lengths),) and 1 <= len(lengths) <= self.max_batch
        self.calls.append(lengths)
        return torch.cat([RampCodec.decode_code(self, x[None, None, :])[0, 0] for x in torch.split(codes, lengths)])


@pytest.mark.parametrize("frames_per_chunk", [25, 50])
def test_stream_batch_ragged_codec_matches_reference_window_plan(frames_per_chunk):
    """infer_stream_batch with a ragged codec: regular windows and tails of a round share codec calls of at most
    max_batch windows, and every utterance still gets exactly the audio of the single-utterance reference procedure."""
    tts, tok = _tts()
    codec = RaggedRampCodec()
    hop = codec.hop
    tts.codec, tts.hop_length = codec, hop
    tts.streaming_frames_per_chunk = frames_per_chunk
    tts.streaming_stride_samples = frames_per_chunk * hop
    rng = np.random.default_rng(5)
    n_gens, n_refs = [143, 9, 260, 61, 230], [60, 75, 52, 20, 60]
    refs = [rng.integers(0, 65536, n).tolist() for n in n_refs]
    kept = [rng.integers(0, 65536, n).tolist() for n in n_gens]
    lm = FakeBatchStreamLM([[tok.speech_base + c for c in k] for k in kept])
    tts.backbone = lm
    got = [[] for _ in refs]
    for out in tts.infer_stream_batch(["hello"] * 5, refs, ["ref"] * 5):
        for b, o in enumerate(out):
            if o is not None:
                got[b].append(o)
    n_windows = 0
    for b in range(5):
        allc = refs[b] + kept[b]
        frames = []
        for (t0, t1, s0, s1) in SO.chunk_plan(len(refs[b]), len(allc), hop=hop, frames=frames_per_chunk):
            wav = RampCodec.decode_code(codec, torch.tensor(allc[t0:t1])[None, None, :])[0, 0].numpy()
            frames.append(wav[s0:s1] if s1 is not None else wav[max(s0, 0):])
        n_windows += len(frames)
        want = SO.linear_overlap_add(frames, tts.streaming_stride_samples) if frames else np.zeros(0, np.float32)
        have = np.concatenate(got[b]) if got[b] else np.zeros(0, np.float32)
        assert have.shape == want.shape, (b, have.shape, want.shape)
        assert np.abs(have - want).max() < 1e-5, b
    assert sum(len(c) for c in codec.calls) == n_windows
    assert any(len(set(c)) > 1 for c in codec.calls)        # windows of different lengths shared a call
