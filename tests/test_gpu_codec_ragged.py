"""GPU: one codec pass over utterances of different lengths (``CodecDecoder.decode_code_ragged`` ->
``nt_codec_decode_ragged``).  Every item must decode as it would alone: against the CPU restatement
(oracle/codec_oracle.py) at the bars of tests/test_gpu_codec.py, and against a batch-1 ``decode_code`` within the
batch-invariance bar.  Equal lengths must reproduce ``decode_code`` bit for bit."""
import numpy as np
import pytest
import torch

from oracle import codec_oracle as CO
from oracle import stream_oracle as SO
from tests.helpers import make_codec, max_err
from tests.test_gpu_facade import _tts

pytestmark = pytest.mark.gpu


def _rms(x):
    return float(x.double().pow(2).mean().sqrt())


def _pack(lengths, codebook, seed):
    g = torch.Generator().manual_seed(seed)
    items = [torch.randint(0, codebook, (n,), generator=g) for n in lengths]
    return items, torch.cat(items)


def _unpack(pcm, lengths, hop):
    return torch.split(pcm.cpu(), [hop * n for n in lengths])


@pytest.mark.parametrize("precision", ["tf32", "mixed", "3xtf32"])
def test_ragged_tiny_config(cuda, precision):
    cfg = CO.CodecConfig.tiny()
    w = CO.random_weights(cfg, 3)
    lengths = (77, 1, 129, 2, 40)
    dec = make_codec(cfg, w, max_batch=5, max_frames=129, precision=precision)
    items, flat = _pack(lengths, cfg.codebook_size, 0)
    pcm = dec.decode_code_ragged(flat, lengths)
    assert pcm.shape == (cfg.hop * sum(lengths),) and pcm.dtype == torch.float32 and pcm.device == dec.device
    for n, c, got in zip(lengths, items, _unpack(pcm, lengths, cfg.hop)):
        with torch.no_grad():
            ref = CO.decode_code(c[None, None, :], w, cfg)[0, 0]
        err = _rms(got - ref)
        assert err < 5e-3 * _rms(ref), (precision, n, err, _rms(ref))
        solo = dec.decode_code(c[None, None, :])[0, 0].cpu()
        assert max_err(got, solo) < 1e-5, (precision, n)
    assert torch.equal(pcm, dec.decode_code_ragged(flat, lengths))        # bit-reproducible run to run


@pytest.mark.parametrize("precision", ["tf32", "3xtf32"])
def test_ragged_uniform_lengths_is_decode_code(cuda, precision):
    cfg = CO.CodecConfig.tiny()
    w = CO.random_weights(cfg, 5)
    dec = make_codec(cfg, w, max_batch=4, max_frames=128, precision=precision)
    codes = torch.randint(0, cfg.codebook_size, (4, 1, 93), generator=torch.Generator().manual_seed(2))
    want = dec.decode_code(codes).reshape(-1)
    got = dec.decode_code_ragged(codes.reshape(-1), [93] * 4)
    assert torch.equal(got, want)


def test_ragged_full_size_3xtf32(cuda):
    cfg = CO.CodecConfig()
    w = CO.random_weights(cfg, 0)
    lengths = (250, 37, 180)
    dec = make_codec(cfg, w, max_batch=3, max_frames=256)
    items, flat = _pack(lengths, 65536, 1)
    pcm = dec.decode_code_ragged(flat.cuda(), lengths)
    assert torch.isfinite(pcm).all()
    for n, c, got in zip(lengths, items, _unpack(pcm, lengths, cfg.hop)):
        with torch.no_grad():
            ref = CO.decode_code(c[None, None, :], w, cfg)[0, 0]
        err, level = _rms(got - ref), _rms(ref)
        print(f"CODEC-RAGGED full size, item of {n} frames: PCM RMS {level:.3f}, abs RMS error {err:.3e}")
        assert 0.02 < level < 0.5, (n, level)
        assert err < 1e-3, (n, err, level)
        solo = dec.decode_code(c[None, None, :].cuda())[0, 0].cpu()
        assert max_err(got, solo) < 1e-5, n


def test_ragged_validation_launches_nothing(cuda):
    cfg = CO.CodecConfig.tiny()
    dec = make_codec(cfg, CO.random_weights(cfg, 4), max_batch=3, max_frames=64)
    L = dec.L
    torch.cuda.synchronize()
    n0 = L.nt_launch_count()
    bad = [
        (torch.zeros(5, dtype=torch.long), [2, 0, 3]),                              # a length of 0
        (torch.zeros(67, dtype=torch.long), [2, 65]),                               # max_frames + 1
        (torch.zeros(4, dtype=torch.long), [1, 1, 1, 1]),                           # max_batch + 1 items
        (torch.full((4,), cfg.codebook_size, dtype=torch.long), [4]),               # id out of range (CPU input)
        (torch.zeros(0, dtype=torch.long), []),                                     # no items
    ]
    for codes, lengths in bad:
        with pytest.raises(ValueError):
            dec.decode_code_ragged(codes, lengths)
    assert L.nt_launch_count() == n0


def _count_codec_calls(dec):
    calls = {"ragged": [], "decode_code": 0}
    ragged, plain = dec.decode_code_ragged, dec.decode_code

    def count_ragged(codes, lengths, validate=None):
        calls["ragged"].append(list(lengths))
        return ragged(codes, lengths, validate)

    def count_plain(codes, validate=None):
        calls["decode_code"] += 1
        return plain(codes, validate)

    dec.decode_code_ragged, dec.decode_code = count_ragged, count_plain
    return calls, plain


def test_facade_infer_batch_uses_one_ragged_call_per_chunk(cuda):
    tts, ccfg = _tts(max_batch=3, seed=23)
    assert tts.watermarker is None
    texts = ["alpha", "beta gamma", "delta epsilon zeta", "eta", "theta iota"]
    refs = [torch.arange(10 + 7 * i) for i in range(5)]
    rts = ["one", "two words", "three", "four", "five"]
    calls, plain = _count_codec_calls(tts.codec)
    wavs = tts.infer_batch(texts, refs, rts)
    prompts = [tts._apply_chat_template(c, rt, t) for t, c, rt in zip(texts, refs, rts)]
    codes = []
    for j in range(0, len(prompts), 3):                     # infer_batch's chunks, same seed and slot base
        codes += [tts._ids_to_codes(g) for g in tts._generate_ids(prompts[j: j + 3], slot_base=j)]
    lengths = [len(c) for c in codes]
    print(f"CODEC-RAGGED facade: kept code lengths {lengths}, codec calls {calls['ragged']}")
    assert len(set(lengths)) > 1                              # the utterances really differ in length
    assert calls["decode_code"] == 0
    assert calls["ragged"] == [lengths[:3], lengths[3:]]
    for c, wav in zip(codes, wavs):
        solo = plain(c[None, None, :])[0, 0].cpu()
        assert wav.shape == (ccfg.hop * len(c),)
        assert max_err(torch.from_numpy(wav), solo) < 1e-5


@pytest.mark.parametrize("F", [25, 50])
def test_facade_stream_batch_ragged_matches_windowed_oracle(cuda, F):
    """infer_stream_batch with the ragged codec: all windows of a round, tails included, share codec calls; the streamed
    PCM of every slot still equals the reference's windowed decode + overlap-add (oracle/stream_oracle.py)."""
    B = 3
    tts, ccfg = _tts(max_batch=B, seed=11)
    cw = CO.random_weights(ccfg, 2)
    hop = ccfg.hop
    tts.hop_length = hop
    tts.streaming_frames_per_chunk = F
    tts.streaming_stride_samples = F * hop
    calls, _ = _count_codec_calls(tts.codec)
    refs = [list(range(60 + 9 * b, 120 + 20 * b)) for b in range(B)]
    texts = ["streaming test sentence number %d" % b for b in range(B)]
    got = [[] for _ in range(B)]
    for out in tts.infer_stream_batch(texts, refs, ["reference"] * B):
        for b, o in enumerate(out):
            if o is not None:
                got[b].append(o)
    assert calls["decode_code"] == 0 and calls["ragged"]
    assert all(len(c) <= B for c in calls["ragged"])
    lm = tts.backbone
    ngen = lm.n_generated[:B].cpu().tolist()
    n_windows = 0
    for b in range(B):
        gen = tts._ids_to_codes(lm.out_tokens[b, : ngen[b]].cpu()).tolist()
        allc = refs[b] + gen
        frames = []
        for (t0, t1, s0, s1) in SO.chunk_plan(len(refs[b]), len(allc), hop=hop, frames=F):
            with torch.no_grad():
                wav = CO.decode_code(torch.tensor(allc[t0:t1])[None, None, :], cw, ccfg)[0, 0].numpy()
            frames.append(wav[s0:s1] if s1 is not None else wav[max(s0, 0):])
        n_windows += len(frames)
        have = np.concatenate(got[b]) if got[b] else np.zeros(0, np.float32)
        if not frames:
            assert have.size == 0
            continue
        want = SO.linear_overlap_add(frames, F * hop)
        assert have.shape == want.shape, (b, have.shape, want.shape, len(gen))
        err = float(np.sqrt(np.mean((have - want) ** 2)) / max(np.sqrt(np.mean(want ** 2)), 1e-9))
        print(f"CODEC-RAGGED stream F={F} slot {b}: {len(gen)} generated frames, {len(frames)} windows, relRMS {err:.2e}")
        assert err < 5e-3, (b, err)
    print(f"CODEC-RAGGED stream F={F}: codec calls (window lengths) {calls['ragged']}")
    assert sum(len(c) for c in calls["ragged"]) == n_windows
