"""CPU: host-side logic above the C-ABI — prompt construction, code<->token mapping, streaming
cross-fade, KV page pool, weight packing, checkpoint reading, sharding plan.  A fake tokenizer /
phonemizer stands in for the HF tokenizer and espeak (neither is available offline)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import stream_oracle as SO


class FakeTokenizer:
    """Character-level tokenizer with the special tokens the reference adds (TRAINING.md:33-57)."""
    SPECIALS = ["<|TEXT_REPLACE|>", "<|TEXT_PROMPT_START|>", "<|TEXT_PROMPT_END|>", "<|SPEECH_REPLACE|>",
                "<|SPEECH_GENERATION_START|>", "<|SPEECH_GENERATION_END|>"]

    def __init__(self, n_speech=65536):
        self.chars = {chr(c): c for c in range(32, 1024)}
        self.chars["\n"] = 10
        self.special_base = 2000
        self.speech_base = 3000
        self.n_speech = n_speech

    def convert_tokens_to_ids(self, tok):
        if tok in self.SPECIALS:
            return self.special_base + self.SPECIALS.index(tok)
        if tok.startswith("<|speech_"):
            return self.speech_base + int(tok[9:-2])
        raise KeyError(tok)

    def encode(self, text, add_special_tokens=True):
        import re

        out = []
        for part in re.split(r"(<\|[A-Za-z_0-9]+\|>)", text):
            if not part:
                continue
            if part.startswith("<|") and part.endswith("|>"):
                out.append(self.convert_tokens_to_ids(part))
            else:
                out += [self.chars[c] for c in part]
        return out

    def decode(self, ids, add_special_tokens=False):
        inv = {v: k for k, v in self.chars.items()}
        s = ""
        for i in ids:
            if i >= self.speech_base:
                s += f"<|speech_{i - self.speech_base}|>"
            elif i >= self.special_base:
                s += self.SPECIALS[i - self.special_base]
            else:
                s += inv[i]
        return s


class FakePhonemizer:
    def phonemize(self, texts):
        return [t.lower().replace(",", " ,") for t in texts]


class FakeCodec:
    device = torch.device("cpu")
    max_batch = 4

    def decode_code(self, codes):
        return torch.zeros(codes.shape[0], 1, 480 * codes.shape[2]) + codes[:, :, :1].float() / 65536.0


class FakeBackbone:
    """transformers-style .generate(): appends fixed ids (some non-speech) and EOS."""
    device = torch.device("cpu")

    def __init__(self, tail):
        self.tail = tail

    def generate(self, ids, **kw):
        self.kw = kw
        return torch.cat((ids, torch.tensor([self.tail])), dim=1)


def _tts(tail=None):
    from neutts import NeuTTS

    tok = FakeTokenizer()
    tail = tail if tail is not None else [tok.speech_base + 5, 65, tok.speech_base + 70000, tok.speech_base + 9, tok.special_base + 5]
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return NeuTTS(tokenizer=tok, phonemizer=FakePhonemizer(), backbone=FakeBackbone(tail), codec=FakeCodec()), tok


def _reference_template(tok, phon, ref_codes, ref_text, input_text):
    """Restatement of neutts/neutts.py:303-332 (the id sequence the facade must reproduce)."""
    to_ph = lambda t: " ".join(phon.phonemize([t])[0].split())
    text = to_ph(ref_text) + " " + to_ph(input_text)
    input_ids = tok.encode(text, add_special_tokens=False)
    ids = tok.encode("user: Convert the text to speech:<|TEXT_REPLACE|>\nassistant:<|SPEECH_REPLACE|>")
    i = ids.index(tok.convert_tokens_to_ids("<|TEXT_REPLACE|>"))
    ids = ids[:i] + [tok.convert_tokens_to_ids("<|TEXT_PROMPT_START|>")] + input_ids + [tok.convert_tokens_to_ids("<|TEXT_PROMPT_END|>")] + ids[i + 1:]
    j = ids.index(tok.convert_tokens_to_ids("<|SPEECH_REPLACE|>"))
    codes = tok.encode("".join(f"<|speech_{c}|>" for c in ref_codes), add_special_tokens=False)
    return ids[:j] + [tok.convert_tokens_to_ids("<|SPEECH_GENERATION_START|>")] + codes


def test_facade_attributes_and_prompt_template():
    tts, tok = _tts()
    assert (tts.sample_rate, tts.max_context, tts.hop_length) == (24000, 2048, 480)
    assert (tts.streaming_overlap_frames, tts.streaming_frames_per_chunk, tts.streaming_lookforward, tts.streaming_lookback,
            tts.streaming_stride_samples) == (1, 25, 5, 50, 12000)
    assert tts._is_quantized_model is False and tts._is_onnx_codec is False
    ref = torch.tensor([5, 17, 65535, 0], dtype=torch.int32)
    for codes in (ref, ref.numpy(), ref.tolist()):
        got = tts._apply_chat_template(codes, "Hello, there", "General  Kenobi")
        assert got == _reference_template(tok, tts.phonemizer, ref.tolist(), "Hello, there", "General  Kenobi")


def test_facade_infer_drops_non_speech_tokens_and_returns_pcm():
    tts, tok = _tts()
    wav = tts.infer("Testing.", torch.tensor([1, 2, 3]), "ref text")
    # the reference's own assertions (tests/test_neutts.py:55-58)
    assert isinstance(wav, np.ndarray) and len(wav) > 0 and not np.isnan(wav).any() and wav.dtype in (np.float32, np.float64)
    assert len(wav) == 480 * 2                   # 65 (text), speech_70000 (out of range) and EOS were dropped
    assert tts.backbone.kw["max_length"] == 2048 and tts.backbone.kw["top_k"] == 50 and tts.backbone.kw["min_new_tokens"] == 50
    assert tts.backbone.kw["temperature"] == 1.0 and tts.backbone.kw["do_sample"] is True
    # string protocol of the seams
    s = tts._infer_torch(tts._apply_chat_template([1], "a", "b"))
    assert s.startswith("<|speech_5|>A<|speech_70000|><|speech_9|>")
    assert len(tts._decode("<|speech_12|>junk<|speech_7|>")) == 960
    with pytest.raises(ValueError, match="No valid speech tokens"):
        tts._decode("no codes here")
    tts2, tok2 = _tts(tail=[65, 66, tok.special_base + 5])
    with pytest.raises(ValueError, match="No valid speech tokens"):
        tts2.infer("x", [1], "y")


def test_facade_rejects_unsupported_backends():
    from neutts import NeuTTS
    from neuttsair import NeuTTSAir

    assert issubclass(NeuTTSAir, NeuTTS)
    kw = dict(tokenizer=FakeTokenizer(), phonemizer=FakePhonemizer())
    with pytest.raises(ValueError, match="GGUF"):
        NeuTTS(backbone_repo="neuphonic/neutts-air-q4-gguf", codec=FakeCodec(), **kw)
    # the reference's own default device strings are accepted (examples/basic_example.py:12-17): "cpu" means host
    # outputs; the engine itself needs CUDA and says so when there is none -- it never falls back to a CPU path
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            NeuTTS(backbone_repo="neuphonic/neutts-air", backbone_device="cpu", codec=FakeCodec(), **kw)
    with pytest.raises(ValueError, match="unsupported backbone_device"):
        NeuTTS(backbone_repo="neuphonic/neutts-air", backbone_device="meta", codec=FakeCodec(), **kw)
    with pytest.raises(ValueError, match="Invalid codec repo"):
        NeuTTS(backbone=FakeBackbone([1]), codec_repo="someone/else", **kw)
    with pytest.raises(ValueError, match="ONNX"):
        NeuTTS(backbone=FakeBackbone([1]), codec_repo="neuphonic/neucodec-onnx-decoder", **kw)


def test_crossfade_equals_reference_overlap_add():
    from neutts.neutts import _CrossFade

    rng = np.random.default_rng(0)
    frames = [rng.standard_normal(12960).astype(np.float32) for _ in range(5)] + [rng.standard_normal(7000).astype(np.float32)]
    fade, out = _CrossFade(12000), []
    for i, f in enumerate(frames):
        out.append(fade.push(f, final=(i == len(frames) - 1)))
    assert [len(o) for o in out[:-1]] == [12000] * 5
    got = np.concatenate(out)
    want = SO.linear_overlap_add(frames, 12000)
    assert got.shape == want.shape and np.abs(got - want).max() < 1e-6


def test_page_pool_and_weight_packing():
    from neutts_air_b200.lm import LMShape, PagePool, _rope_pair_perm, pack_weights
    from oracle import lm_oracle as LO
    from tests.helpers import lm_state_dict

    pool = PagePool(8, shuffle_seed=1)
    a = pool.alloc(3)
    b = pool.alloc(5)
    assert sorted(a + b) == list(range(8))
    with pytest.raises(RuntimeError):
        pool.alloc(1)
    pool.release(a)
    assert sorted(pool.alloc(3)) == sorted(a)
    assert _rope_pair_perm(2)[:6].tolist() == [0, 32, 1, 33, 2, 34] and _rope_pair_perm(2)[64:68].tolist() == [64, 96, 65, 97]
    cfg = LO.LMConfig.tiny()
    w = LO.random_weights(cfg, 0)
    shape = LMShape(cfg.vocab_size, cfg.hidden_size, cfg.intermediate_size, cfg.num_layers, cfg.num_heads, cfg.num_kv_heads)
    pk = pack_weights(shape, lm_state_dict(w), "cpu")
    L0 = w.layers[0]
    assert pk["wqkv"][0].shape == ((cfg.num_heads + 2 * cfg.num_kv_heads) * 64, cfg.hidden_size)
    assert torch.equal(pk["wqkv"][0][1].float(), L0["wq"][32].bfloat16().float())              # partner row adjacent
    assert torch.equal(pk["wqkv"][0][cfg.num_heads * 64 + 2].float(), L0["wk"][1].bfloat16().float())
    assert torch.equal(pk["wqkv"][0][-1].float(), L0["wv"][-1].bfloat16().float())              # v rows keep natural order
    assert torch.equal(pk["bqkv"][0][:4], torch.stack((L0["bq"][0], L0["bq"][32], L0["bq"][1], L0["bq"][33])))
    assert torch.equal(pk["wgu"][0][0].float(), L0["wg"][0].bfloat16().float()) and torch.equal(pk["wgu"][0][1].float(), L0["wu"][0].bfloat16().float())
    assert pk["lm_head"] is pk["embed"]


def test_loader_reads_hf_checkpoint(tmp_path, monkeypatch):
    pytest.importorskip("transformers")
    monkeypatch.setenv("HF_HUB_OFFLINE", "1")        # the missing-repo lookup below stays in the local HF cache
    from neutts_air_b200 import loader
    from neutts_air_b200.lm import LMShape
    from oracle import lm_oracle as LO

    cfg = LO.LMConfig.tiny()
    w = LO.random_weights(cfg, 2)
    LO.to_hf_model(cfg, w).save_pretrained(tmp_path)
    hf_cfg = json.loads((tmp_path / "config.json").read_text())
    shape = LMShape.from_hf_config(hf_cfg)
    assert (shape.vocab_size, shape.hidden_size, shape.num_layers, shape.num_heads, shape.num_kv_heads, shape.head_dim) == \
        (cfg.vocab_size, cfg.hidden_size, cfg.num_layers, cfg.num_heads, cfg.num_kv_heads, 64)
    assert shape.rope_theta == 1e6 and shape.tie_embeddings
    sd = loader.read_state_dict(loader.resolve_repo(str(tmp_path)))
    assert torch.equal(sd["model.layers.1.mlp.down_proj.weight"], w.layers[1]["wd"])
    with pytest.raises(FileNotFoundError):
        loader.resolve_repo("definitely/not-a-repo-xyz")


def test_codec_loader_key_mapping_and_packing():
    from neutts_air_b200 import loader
    from neutts_air_b200.codec import CodecShape, idft_basis, pack_weights
    from oracle import codec_oracle as CO

    cfg = CO.CodecConfig.tiny()
    w = CO.random_weights(cfg, 1)
    sd = {"generator.quantizer.project_out.weight": w.project_out_w, "generator.quantizer.project_out.bias": w.project_out_b,
          "fc_post_a.weight": w.fc_post_a_w, "fc_post_a.bias": w.fc_post_a_b,
          "generator.backbone.embed.weight": w.embed_w, "generator.backbone.embed.bias": w.embed_b,
          "generator.backbone.final_layer_norm.weight": w.final_ln_w, "generator.backbone.final_layer_norm.bias": w.final_ln_b,
          "generator.head.out.weight": w.head_w, "generator.head.out.bias": w.head_b}
    names = dict(n1w="norm1.weight", n1b="norm1.bias", c1w="conv1.weight", c1b="conv1.bias", n2w="norm2.weight", n2b="norm2.bias",
                 c2w="conv2.weight", c2b="conv2.bias")
    for grp, blocks in (("prior_net", w.prior), ("post_net", w.post)):
        for i, r in enumerate(blocks):
            for k, v in r.items():
                sd[f"generator.backbone.{grp}.{i}.{names[k]}"] = v
    for i, b in enumerate(w.blocks):
        p = f"generator.backbone.transformers.{i}."
        sd.update({p + "att_norm.weight": b["att_norm"], p + "att.c_attn.weight": b["wqkv"], p + "att.c_proj.weight": b["wproj"],
                   p + "ffn_norm.weight": b["ffn_norm"], p + "mlp.fc1.weight": b["fc1"], p + "mlp.fc2.weight": b["fc2"]})
    shape, wd = loader.codec_weights_from_state_dict(sd)
    assert (shape.hidden, shape.depth, shape.heads, shape.n_fft, shape.hop, shape.quant_dim) == (128, 2, 2, 64, 16, 64)
    pk = pack_weights(shape, wd, "cpu")
    # collapsed FSQ affine == fc_post_a(project_out(z)) on every digit vector
    z = CO.fsq_dequant(torch.arange(0, 65536, 257), cfg)
    want = (z @ w.project_out_w.T + w.project_out_b) @ w.fc_post_a_w.T + w.fc_post_a_b
    assert float((z @ pk["fsq_w"].T + pk["fsq_b"] - want).abs().max()) < 1e-5
    # tap-major conv flattening
    assert torch.equal(pk["embed_w"][3, 2 * 128 + 5], w.embed_w[3, 5, 2])
    # windowed inverse-rDFT basis reproduces irfft * hann
    g = torch.Generator().manual_seed(0)
    nb = 33
    spec = torch.complex(torch.randn(4, nb, generator=g), torch.randn(4, nb, generator=g))
    B = idft_basis(64, 96)
    got = torch.cat((spec.real, spec.imag), 1) @ B[:, :2 * nb].T
    ref = torch.fft.irfft(spec, 64, dim=1) * torch.hann_window(64)
    assert float((got - ref).abs().max()) < 1e-5 and float(B[:, 2 * nb:].abs().max()) == 0.0


def test_shard_plan_is_a_balanced_partition():
    from neutts_air_b200 import dist

    lens = [700, 210, 1400, 333, 900, 901, 250, 1111, 640]
    for ws in (1, 2, 4, 8):
        plan = dist.shard_plan(len(lens), lens, ws)
        assert sorted(i for p in plan for i in p) == list(range(len(lens)))
        assert max(len(p) for p in plan) - min(len(p) for p in plan) <= 1
    loads = [sum(lens[i] for i in p) for p in dist.shard_plan(len(lens), lens, 2)]
    assert max(loads) / min(loads) < 1.25


class FakeStreamLM:
    """prefill()/decode() surface of SpeechLM with a scripted token stream (speech ids, junk ids, EOS)."""
    device = torch.device("cpu")

    def __init__(self, script, max_new=4096):
        self.script, self.max_new = list(script), max_new
        self.out_tokens = torch.zeros(1, max_new, dtype=torch.int32)
        self.n_generated = torch.zeros(1, dtype=torch.int32)
        self.done = torch.zeros(1, dtype=torch.int32)
        self.decode_calls = []

    def sampling(self, eos, min_new, max_new, top_k, temperature, seed):
        self.eos, self.limit = eos, max_new
        return None

    def _emit(self):
        n = int(self.n_generated[0])
        if int(self.done[0]) or n >= self.limit:
            return
        tok = self.script[n] if n < len(self.script) else self.eos
        self.out_tokens[0, n] = tok
        self.n_generated[0] = n + 1
        if tok == self.eos or n + 1 >= self.limit:
            self.done[0] = 1

    def prefill(self, prompts, sp):
        self._emit()

    def decode(self, steps, sp):
        assert steps >= 1
        self.decode_calls.append(steps)
        for _ in range(steps):
            self._emit()


class RampCodec:
    """Deterministic 'codec': frame i of the window becomes hop samples of code/1000 + 0.01 * position-in-window,
    so a wrong window start, slice or cross-fade weight changes the output."""
    device = torch.device("cpu")
    max_batch = 1
    hop = 8

    def decode_code(self, codes):
        c = codes[0, 0].float()
        frames = c[:, None] / 1000.0 + 0.01 * torch.arange(len(c))[:, None] + torch.zeros(1, self.hop)
        return frames.reshape(1, 1, -1)


@pytest.mark.parametrize("n_gen,junk_every,limit", [(143, 0, None), (90, 7, None), (30, 0, None), (12, 3, None), (400, 5, 301)])
def test_stream_matches_reference_window_plan(n_gen, junk_every, limit):
    """infer_stream == the reference's window bookkeeping (neutts/neutts.py:373-465) restated in
    oracle/stream_oracle.py: same codec windows, same slices, same triangular cross-fade, including the
    ragged tail, non-speech ids interleaved in the stream, and a stop by max_length instead of EOS."""
    tts, tok = _tts()
    codec = RampCodec()
    hop = codec.hop
    tts.codec, tts.hop_length = codec, hop
    tts.streaming_stride_samples = tts.streaming_frames_per_chunk * hop
    rng = np.random.default_rng(n_gen)
    gen_codes = rng.integers(0, 65536, n_gen).tolist()
    script = []
    for i, c in enumerate(gen_codes):
        if junk_every and i % junk_every == 0:
            script.append(65)                       # a text token in the middle of speech: dropped
        script.append(tok.speech_base + c)
    lm = FakeStreamLM(script)
    tts.backbone = lm
    ref_codes = rng.integers(0, 65536, 60).tolist()
    if limit is not None:
        prompt_len = len(tts._apply_chat_template(ref_codes, "ref", "hello"))
        tts.max_context = prompt_len + limit
        kept = [t - tok.speech_base for t in script[:limit] if t >= tok.speech_base]
    else:
        kept = gen_codes
    chunks = list(tts.infer_stream("hello", ref_codes, "ref"))
    if limit is not None:
        assert int(lm.n_generated[0]) == limit      # stopped by max_length, not EOS
    # expected: decode every planned window with the same codec, slice, overlap-add
    allc = ref_codes + kept
    frames = []
    for (t0, t1, s0, s1) in SO.chunk_plan(len(ref_codes), len(allc), hop=hop):
        wav = codec.decode_code(torch.tensor(allc[t0:t1])[None, None, :])[0, 0].numpy()
        frames.append(wav[s0:s1] if s1 is not None else wav[max(s0, 0):])
    want = SO.linear_overlap_add(frames, tts.streaming_stride_samples) if frames else np.zeros(0, np.float32)
    got = np.concatenate(chunks) if chunks else np.zeros(0, np.float32)
    assert got.shape == want.shape
    assert np.abs(got - want).max() < 1e-5
    assert all(len(c) == tts.streaming_stride_samples for c in chunks[:-1])
    assert max(lm.decode_calls, default=0) <= tts.streaming_frames_per_chunk + tts.streaming_lookforward


def test_reference_signature_defaults():
    """Constructor signature == the reference's (neutts/neutts.py:75-81) for the four positional parameters."""
    import inspect

    from neutts import NeuTTS

    sig = inspect.signature(NeuTTS.__init__)
    got = [(n, p.default) for n, p in list(sig.parameters.items())[1:5]]
    assert got == [("backbone_repo", "neuphonic/neutts-nano"), ("backbone_device", "cpu"),
                   ("codec_repo", "neuphonic/neucodec"), ("codec_device", "cpu")]


EXAMPLE_CALLS = os.path.join(os.path.dirname(__file__), "golden", "basic_example_calls.json")


def test_reference_basic_example_runs_unmodified(tmp_path, monkeypatch):
    """SURVEY §8c golden (4): the calls the reference's examples/basic_example.py makes when it runs unmodified
    (recorded by oracle/record_example_calls.py into tests/golden/basic_example_calls.json) drive THIS repo's
    ``neutts.NeuTTS`` (ctor with the reference's device strings, encode_reference, infer, soundfile.write) and
    write a wav of 480 * N samples.  Checkpoints, tokenizer and espeak do not exist offline, so the three loaders
    are replaced by the fakes of this file; the facade runs unmodified."""
    import importlib

    import neutts.neutts as NN

    trace = json.load(open(EXAMPLE_CALLS))
    assert [c["call"] for c in trace["calls"]] == ["neutts.NeuTTS", "NeuTTS.encode_reference", "NeuTTS.infer", "soundfile.write"]
    written = {}

    def sf_write(path, wav, sr):
        written.update(path=path, wav=np.asarray(wav), sr=sr)

    tok = FakeTokenizer()
    tail = [tok.speech_base + c for c in (5, 9, 11, 70000, 13)] + [65, tok.special_base + 5]   # 4 valid codes, junk, EOS
    seen = {}

    def load_backbone(self, repo, device, backbone=None):
        seen["backbone"] = (repo, device)
        self.tokenizer = tok
        self.backbone = FakeBackbone(tail)

    def load_codec(self, repo, device, codec=None):
        seen["codec"] = (repo, device)
        self.codec = FakeCodec()

    monkeypatch.setattr(NN.NeuTTS, "_load_backbone", load_backbone)
    monkeypatch.setattr(NN.NeuTTS, "_load_codec", load_codec)
    monkeypatch.setattr(NN.NeuTTS, "_load_phonemizer", staticmethod(lambda: FakePhonemizer()))
    # reference voice: audio file + the pre-encoded codes next to it, as the reference ships them (samples/dave.{wav,pt})
    (tmp_path / "dave.wav").write_bytes(b"RIFF....WAVE")
    torch.save(torch.tensor([54, 65493, 7], dtype=torch.int32), tmp_path / "dave.pt")
    for name, text in trace["files"].items():
        (tmp_path / name).write_text(text)
    rets = []

    def arg(v):
        if isinstance(v, dict) and "$ret" in v:
            return rets[v["$ret"]]
        return v.replace("{tmp}", str(tmp_path)) if isinstance(v, str) else v

    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for c in trace["calls"]:
            args, kwargs = [arg(a) for a in c["args"]], {k: arg(v) for k, v in c["kwargs"].items()}
            if c["call"] == "neutts.NeuTTS":
                cls = importlib.import_module("neutts").NeuTTS   # `from neutts import NeuTTS` resolves to this repo's package
                assert cls is NN.NeuTTS
                tts = cls(*args, **kwargs)
                rets.append(tts)
            elif c["call"] == "soundfile.write":
                rets.append(sf_write(*args, **kwargs))
            else:
                rets.append(getattr(tts, c["call"].split(".", 1)[1])(*args, **kwargs))
    assert seen == {"backbone": ("neuphonic/neutts-air", "cpu"), "codec": ("neuphonic/neucodec", "cpu")}
    assert written["sr"] == 24000 and written["path"].endswith("out.wav")
    assert written["wav"].dtype == np.float32 and written["wav"].shape == (480 * 4,) and np.isfinite(written["wav"]).all()


def test_generate_batch_caps_are_per_sequence():
    """ADVICE r1: max_length is prompt + generated PER SEQUENCE -- a long prompt must not shorten its neighbours."""
    from neutts_air_b200.lm import SpeechLM

    calls = {}

    class Stub(SpeechLM):
        def __init__(self):
            self.max_ctx, self.max_new, self.max_batch, self.device = 2048, 2048, 2, torch.device("cpu")
            self.n_generated = torch.tensor([5, 7])
            self.out_tokens = torch.zeros(2, 2048, dtype=torch.int32)
            self.done = torch.ones(2, dtype=torch.int32)

        def sampling(self, *a, **kw):
            calls["sampling"] = (a, kw)
            return types.SimpleNamespace(max_new_tokens=a[2])

        def prefill(self, prompts, sp):
            calls["prefill"] = [len(p) for p in prompts]

        def decode(self, n, sp):
            calls["decode"] = calls.get("decode", 0) + n

    import types
    lm = Stub()
    lm.generate_batch([[1] * 1500, [2] * 300], eos_token_id=9, max_length=2048, check_every=4096)
    a, kw = calls["sampling"]
    assert a[2] == 1748                       # the loop runs to the LARGEST per-sequence budget ...
    assert list(kw["limits"]) == [548, 1748]  # ... and every slot carries its own cap (2048 - prompt length)
    lm.generate_batch([[1] * 300, [2] * 300], eos_token_id=9, max_length=2048, check_every=4096)
    assert calls["sampling"][1]["limits"] is None and calls["sampling"][0][2] == 1748


class FakeBatchStreamLM:
    """Batched prefill()/decode() surface of SpeechLM: one scripted token stream per slot, lock-step decoding,
    finished slots idle (as inside the persistent kernel)."""
    device = torch.device("cpu")

    def __init__(self, scripts, max_new=4096):
        self.scripts, self.max_new = [list(s) for s in scripts], max_new
        B = len(scripts)
        self.out_tokens = torch.zeros(B, max_new, dtype=torch.int32)
        self.n_generated = torch.zeros(B, dtype=torch.int32)
        self.done = torch.zeros(B, dtype=torch.int32)
        self.decode_calls = []

    def sampling(self, eos, min_new, max_new, top_k, temperature, seed, limits=None):
        self.eos = eos
        self.limits = list(limits) if limits is not None else [max_new] * len(self.scripts)
        return None

    def _emit(self):
        for b, script in enumerate(self.scripts):
            n = int(self.n_generated[b])
            if int(self.done[b]) or n >= self.limits[b]:
                continue
            tok = script[n] if n < len(script) else self.eos
            self.out_tokens[b, n] = tok
            self.n_generated[b] = n + 1
            if tok == self.eos or n + 1 >= self.limits[b]:
                self.done[b] = 1

    def prefill(self, prompts, sp):
        self._emit()

    def decode(self, steps, sp):
        assert steps >= 1
        self.decode_calls.append(steps)
        for _ in range(steps):
            self._emit()


class BatchRampCodec(RampCodec):
    max_batch = 2          # smaller than the batch: same-length windows are split over several codec calls

    def decode_code(self, codes):
        assert codes.shape[0] <= self.max_batch
        return torch.cat([RampCodec.decode_code(self, codes[r: r + 1]) for r in range(codes.shape[0])])


@pytest.mark.parametrize("frames_per_chunk", [25, 50])
def test_stream_batch_matches_reference_window_plan_per_utterance(frames_per_chunk):
    """infer_stream_batch (BASELINE configs[4]: batch-8 streaming; 50 = "codec every 50 tokens"): every utterance of
    the batch gets exactly the audio the single-utterance reference procedure gives it -- different reference
    lengths, generated lengths (one ends after 9 tokens, one runs 3x longer), junk ids, one slot stopped by its
    own max_length -- while the slots decode in lock-step and share codec calls."""
    tts, tok = _tts()
    codec = BatchRampCodec()
    hop = codec.hop
    tts.codec, tts.hop_length = codec, hop
    tts.streaming_frames_per_chunk = frames_per_chunk
    tts.streaming_stride_samples = frames_per_chunk * hop
    rng = np.random.default_rng(77)
    n_gens, n_refs, junk = [143, 9, 400, 61, 230], [60, 75, 52, 120, 60], [0, 0, 5, 3, 0]
    refs = [rng.integers(0, 65536, n).tolist() for n in n_refs]
    scripts, kept = [], []
    for n, j in zip(n_gens, junk):
        codes = rng.integers(0, 65536, n).tolist()
        sc = []
        for i, c in enumerate(codes):
            if j and i % j == 0:
                sc.append(65)
            sc.append(tok.speech_base + c)
        scripts.append(sc)
        kept.append(codes)
    lm = FakeBatchStreamLM(scripts)
    tts.backbone = lm
    # slot 2 is cut by max_length: the facade caps it at max_context - len(prompt)
    prompt_lens = [len(tts._apply_chat_template(r, "ref", "hello")) for r in refs]
    tts.max_context = prompt_lens[2] + 301
    lim2 = 301
    kept[2] = [t - tok.speech_base for t in scripts[2][:lim2] if t >= tok.speech_base]
    got = [[] for _ in refs]
    n_yields = 0
    for out in tts.infer_stream_batch(["hello"] * 5, refs, ["ref"] * 5):
        assert len(out) == 5 and any(o is not None for o in out)
        n_yields += 1
        for b, o in enumerate(out):
            if o is not None:
                got[b].append(o)
    assert int(lm.n_generated[2]) == lim2
    for b in range(5):
        allc = refs[b] + kept[b]
        frames = []
        for (t0, t1, s0, s1) in SO.chunk_plan(len(refs[b]), len(allc), hop=hop, frames=frames_per_chunk):
            wav = RampCodec.decode_code(codec, torch.tensor(allc[t0:t1])[None, None, :])[0, 0].numpy()
            frames.append(wav[s0:s1] if s1 is not None else wav[max(s0, 0):])
        want = SO.linear_overlap_add(frames, tts.streaming_stride_samples) if frames else np.zeros(0, np.float32)
        have = np.concatenate(got[b]) if got[b] else np.zeros(0, np.float32)
        assert have.shape == want.shape, (b, have.shape, want.shape)
        assert np.abs(have - want).max() < 1e-5, b
    assert max(lm.decode_calls) <= frames_per_chunk + tts.streaming_lookforward
    assert n_yields < sum(len(g) for g in got)          # rounds are shared between the utterances
