"""Drop-in ``neutts.NeuTTS`` on the B200 engine.

Same public surface as the reference facade (``/root/reference/neutts/neutts.py:73-465``):
constructor signature and attributes (``:75-98``), ``infer`` (``:216``), ``infer_stream`` (``:245``),
``encode_reference`` (``:266``), the private seams ``_apply_chat_template`` / ``_infer_torch`` /
``_decode`` / ``_to_phones``, and the same error convention (``ValueError`` / ``ImportError`` /
``NotImplementedError``).  Behind it, hot path A (speech-LM prefill + decode) and hot path B
(NeuCodec decoder) run in ``libneutts_b200.so`` on an sm_100a GPU; there is no CPU fallback and no
llama.cpp / ONNX / vLLM dispatch.

What differs from the reference, on purpose:
  * generated ids go straight from the device to the codec (``speech id = token id - id(<|speech_0|>)``)
    instead of ``tokenizer.decode`` + regex; ``_infer_torch`` / ``_decode`` still speak the string
    protocol so code written against the reference keeps working;
  * ``infer_batch`` takes lists and shards utterances over ranks (one NCCL all-gather of waveforms);
  * ``infer_stream`` works on this backend (the reference raises for torch backbones) with the
    reference's streaming window geometry (``:87-91``) and an incremental cross-fade;
  * tokenizer, phonemizer, backbone and codec can be injected, so the facade runs offline.
"""
from __future__ import annotations

import re
import warnings
from pathlib import Path
from typing import Generator, Sequence

import numpy as np
import torch

SPEECH_RE = re.compile(r"<\|speech_(\d+)\|>")
CHAT = "user: Convert the text to speech:<|TEXT_REPLACE|>\nassistant:<|SPEECH_REPLACE|>"


def _split_frames(pcm: np.ndarray, lengths: Sequence[int]) -> list:
    """Packed PCM of a ragged codec call -> one waveform per item (hop = samples per frame)."""
    hop = pcm.shape[-1] // sum(lengths)
    return np.split(pcm, np.cumsum([hop * n for n in lengths])[:-1])


class _CrossFade:
    """Incremental equivalent of the reference's ``_linear_overlap_add`` (``neutts/neutts.py:46-70``):
    triangular weights over every chunk, weighted sum / weight sum, but only the samples a new chunk
    can still change are kept (the reference re-sums the whole history on every chunk)."""

    def __init__(self, stride: int):
        self.stride = stride
        self.acc = np.zeros(0, dtype=np.float32)
        self.wsum = np.zeros(0, dtype=np.float32)

    def push(self, frame: np.ndarray, final: bool = False) -> np.ndarray:
        n = frame.shape[-1]
        t = np.linspace(0, 1, n + 2, dtype=np.float32)[1:-1]
        w = np.abs(0.5 - (t - 0.5))
        if n > self.acc.shape[0]:
            grow = n - self.acc.shape[0]
            self.acc = np.concatenate([self.acc, np.zeros(grow, np.float32)])
            self.wsum = np.concatenate([self.wsum, np.zeros(grow, np.float32)])
        self.acc[:n] += w * frame.astype(np.float32)
        self.wsum[:n] += w
        take = self.acc.shape[0] if final else min(self.stride, self.acc.shape[0])
        out = self.acc[:take] / self.wsum[:take]
        self.acc, self.wsum = self.acc[take:], self.wsum[take:]
        return out


class NeuTTS:
    def __init__(self, backbone_repo="neuphonic/neutts-nano", backbone_device="cpu", codec_repo="neuphonic/neucodec",
                 codec_device="cpu", *, tokenizer=None, phonemizer=None, backbone=None, codec=None,
                 max_batch: int = 1, seed: int | None = None):
        """Same positional signature and defaults as the reference (``neutts/neutts.py:75-81``), so
        ``examples/basic_example.py:12-17`` runs unmodified.  The device strings keep their reference
        meaning for the CALLER -- ``"cpu"`` = results come back as host arrays, which this facade always
        does -- but the engines themselves only exist for sm_100a: a ``"cpu"`` request runs on the current
        CUDA device and says so once (there is no CPU fallback)."""
        # constants the reference exposes (neutts/neutts.py:84-91)
        self.sample_rate = 24_000
        self.max_context = 2048
        self.hop_length = 480
        self.streaming_overlap_frames = 1
        self.streaming_frames_per_chunk = 25
        self.streaming_lookforward = 5
        self.streaming_lookback = 50
        self.streaming_stride_samples = self.streaming_frames_per_chunk * self.hop_length
        self._is_quantized_model = False
        self._is_onnx_codec = False
        self.tokenizer = tokenizer
        self.max_batch = max_batch
        self.seed = seed
        self.phonemizer = phonemizer if phonemizer is not None else self._load_phonemizer()
        self._load_backbone(backbone_repo, backbone_device, backbone)
        self._load_codec(codec_repo, codec_device, codec)
        try:  # optional watermark, exactly as the reference (neutts/neutts.py:110-121)
            import perth

            self.watermarker = perth.PerthImplicitWatermarker()
        except (ImportError, AttributeError) as e:
            warnings.warn(f"Perth watermarking unavailable: {e}. Audio will not be watermarked.")
            self.watermarker = None
        self._speech_base = None

    # ------------------------------------------------------------------ loading
    @staticmethod
    def _load_phonemizer():
        try:
            from phonemizer.backend import EspeakBackend
        except ImportError as e:
            raise ImportError("phonemizer (and espeak-ng) are required for text input; "
                              "pass phonemizer=... to NeuTTS to inject one") from e
        return EspeakBackend(language="en-us", preserve_punctuation=True, with_stress=True)

    def _load_backbone(self, backbone_repo, backbone_device, backbone=None):
        if backbone is not None:
            self.backbone = backbone
            return
        if str(backbone_repo).endswith("gguf"):
            raise ValueError("GGUF / llama.cpp backbones are not dispatched by the B200 build; "
                             "use the safetensors checkpoint (e.g. neuphonic/neutts-air)")
        backbone_device = self._engine_device(backbone_device, "backbone")
        from neutts_air_b200 import loader

        if self.tokenizer is None:
            self.tokenizer = loader.load_tokenizer(backbone_repo)
        self.backbone = loader.load_speech_lm(backbone_repo, backbone_device, max_batch=self.max_batch,
                                              max_ctx=self.max_context)

    def _load_codec(self, codec_repo, codec_device, codec=None):
        if codec is not None:
            self.codec = codec
            return
        if str(codec_repo).endswith(".onnx") or codec_repo == "neuphonic/neucodec-onnx-decoder":
            raise ValueError("ONNX codec decoders are not dispatched by the B200 build; use 'neuphonic/neucodec'")
        if codec_repo not in ("neuphonic/neucodec", "neuphonic/distill-neucodec") and not Path(str(codec_repo)).exists():
            raise ValueError("Invalid codec repo! Must be one of: 'neuphonic/neucodec', 'neuphonic/distill-neucodec' "
                             "(or a local checkpoint directory).")
        codec_device = self._engine_device(codec_device, "codec")
        from neutts_air_b200 import loader

        self.codec = loader.load_codec_decoder(codec_repo, codec_device, max_batch=self.max_batch,
                                               max_frames=self.max_context)

    @staticmethod
    def _engine_device(requested, what: str):
        """Reference device string -> the CUDA device the B200 engine runs on."""
        dev = torch.device(requested)
        if dev.type == "cuda":
            return dev
        if dev.type != "cpu":
            raise ValueError(f"unsupported {what}_device {requested!r}")
        if not torch.cuda.is_available():
            raise RuntimeError(f"neutts (B200 build): {what}_device={requested!r} was requested, but the engines exist only for "
                               "CUDA sm_100a and no CUDA device is visible (there is no CPU fallback)")
        warnings.warn(f"neutts (B200 build): {what}_device={requested!r} -> running on cuda:{torch.cuda.current_device()}; "
                      "outputs are returned on the host as with the reference's CPU path", stacklevel=3)
        return torch.device("cuda", torch.cuda.current_device())

    # ------------------------------------------------------------------ prompt construction (N1)
    def _to_phones(self, text: str) -> str:
        return " ".join(self.phonemizer.phonemize([text])[0].split())

    def _tok_id(self, name: str) -> int:
        return self.tokenizer.convert_tokens_to_ids(name)

    @property
    def speech_base(self) -> int:
        """Token id of ``<|speech_0|>``; speech ids are contiguous above it (TRAINING.md:52-57 adds
        them with one ``add_tokens`` call), which is checked once here."""
        if self._speech_base is None:
            base = self._tok_id("<|speech_0|>")
            probe = (1, 4095, 65535)
            if any(self._tok_id(f"<|speech_{i}|>") != base + i for i in probe):
                raise ValueError("tokenizer does not map <|speech_N|> to consecutive ids")
            self._speech_base = base
        return self._speech_base

    def _apply_chat_template(self, ref_codes, ref_text: str, input_text: str) -> list:
        """Same id sequence as the reference builds (``neutts/neutts.py:303-332``):
        ``user: Convert the text to speech: [TPS] phones [TPE] \\nassistant: [SGS] ref speech ids``."""
        phones = self._to_phones(ref_text) + " " + self._to_phones(input_text)
        text_ids = self.tokenizer.encode(phones, add_special_tokens=False)
        ids = list(self.tokenizer.encode(CHAT))
        t = ids.index(self._tok_id("<|TEXT_REPLACE|>"))
        ids = ids[:t] + [self._tok_id("<|TEXT_PROMPT_START|>")] + list(text_ids) + [self._tok_id("<|TEXT_PROMPT_END|>")] + ids[t + 1:]
        s = ids.index(self._tok_id("<|SPEECH_REPLACE|>"))
        codes = [int(c) for c in (ref_codes.tolist() if hasattr(ref_codes, "tolist") else ref_codes)]
        base = self.speech_base
        return ids[:s] + [self._tok_id("<|SPEECH_GENERATION_START|>")] + [base + c for c in codes]

    # ------------------------------------------------------------------ hot path A
    def _generate_ids(self, prompts: Sequence[Sequence[int]], max_new_tokens: int | None = None,
                      min_new_tokens: int = 50, slot_base: int = 0) -> list:
        """Batched device-side generation; returns generated token ids per prompt (CPU int64 tensors).
        Sampling parameters are the reference's (``neutts/neutts.py:338-347``)."""
        eos = self._tok_id("<|SPEECH_GENERATION_END|>")
        seed = self.seed if self.seed is not None else int(torch.randint(0, 2**31 - 1, (1,)).item())
        if hasattr(self.backbone, "generate_batch"):
            return self.backbone.generate_batch(list(prompts), eos, max_length=self.max_context, min_new_tokens=min_new_tokens,
                                                temperature=1.0, top_k=50, max_new_tokens=max_new_tokens, seed=seed,
                                                slot_base=slot_base)
        outs = []  # injected transformers-style backbone: one sequence at a time, as the reference does
        for p in prompts:
            t = torch.tensor(list(p)).unsqueeze(0).to(self.backbone.device)
            with torch.no_grad():
                o = self.backbone.generate(t, max_length=self.max_context, eos_token_id=eos, do_sample=True, temperature=1.0,
                                           top_k=50, use_cache=True, min_new_tokens=min_new_tokens)
            outs.append(o[0, t.shape[-1]:].cpu().long())
        return outs

    def _ids_to_codes(self, ids: torch.Tensor) -> torch.Tensor:
        """Drop every token that is not ``<|speech_N|>`` (the reference's regex does the same, ``:276``)."""
        base = self.speech_base
        n_codes = getattr(getattr(self.codec, "shape", None), "fsq_levels", 4) ** getattr(getattr(self.codec, "shape", None), "fsq_dims", 8)
        c = ids.long() - base
        return c[(c >= 0) & (c < n_codes)]

    def _ids_to_codes_masked(self, ids: torch.Tensor):
        """Tensor form of ``_ids_to_codes`` for the device-side code history: (codes, keep mask), same shape as ids."""
        shape = getattr(self.codec, "shape", None)
        n_codes = getattr(shape, "fsq_levels", 4) ** getattr(shape, "fsq_dims", 8)
        c = ids.long() - self.speech_base
        return c, (c >= 0) & (c < n_codes)

    def _infer_torch(self, prompt_ids: list) -> str:
        """String protocol of the reference seam (``neutts/neutts.py:334-352``)."""
        out = self._generate_ids([prompt_ids])[0]
        return self.tokenizer.decode(out.numpy().tolist(), add_special_tokens=False)

    # ------------------------------------------------------------------ hot path B
    def _decode_codes(self, codes: Sequence[torch.Tensor]) -> list:
        """codes: list of 1-D int tensors -> list of float32 numpy waveforms.  A codec with ``decode_code_ragged`` takes
        up to ``max_batch`` utterances per call in input order, whatever their lengths; any other codec gets one
        ``decode_code`` call per distinct length."""
        out = [None] * len(codes)
        by_len: dict = {}
        for i, c in enumerate(codes):
            if len(c) == 0:
                raise ValueError("No valid speech tokens found in the output.")
            by_len.setdefault(len(c), []).append(i)
        cap = getattr(self.codec, "max_batch", 1)
        if hasattr(self.codec, "decode_code_ragged"):
            for j in range(0, len(codes), cap):
                grp = [codes[i].long().flatten() for i in range(j, min(j + cap, len(codes)))]
                lens = [len(c) for c in grp]
                with torch.no_grad():
                    pcm = self.codec.decode_code_ragged(torch.cat(grp).to(self.codec.device), lens).cpu().numpy()
                out[j: j + len(grp)] = _split_frames(pcm, lens)
            return out
        for n, idxs in by_len.items():
            for j in range(0, len(idxs), cap):
                grp = idxs[j: j + cap]
                batch = torch.stack([codes[i].long() for i in grp])[:, None, :].to(self.codec.device)
                with torch.no_grad():
                    pcm = self.codec.decode_code(batch).cpu().numpy()
                for r, i in enumerate(grp):
                    out[i] = pcm[r, 0, :]
        return out

    def _decode(self, codes) -> np.ndarray:
        """``codes``: the ``<|speech_N|>`` string of the reference seam (``neutts/neutts.py:273-295``) or a 1-D int sequence."""
        if isinstance(codes, str):
            ids = [int(n) for n in SPEECH_RE.findall(codes)]
            codes = torch.tensor(ids, dtype=torch.long)
        else:
            codes = torch.as_tensor(codes, dtype=torch.long).flatten()
        if len(codes) == 0:
            raise ValueError("No valid speech tokens found in the output.")
        return self._decode_codes([codes])[0]

    def _watermark(self, wav: np.ndarray) -> np.ndarray:
        return wav if self.watermarker is None else self.watermarker.apply_watermark(wav, sample_rate=24_000)

    # ------------------------------------------------------------------ public API
    def infer(self, text: str, ref_codes, ref_text: str) -> np.ndarray:
        """Text + reference voice -> 24 kHz float32 waveform (``neutts/neutts.py:216-243``)."""
        return self.infer_batch([text], [ref_codes], [ref_text])[0]

    def infer_from_prompt_ids(self, prompts: Sequence[Sequence[int]], max_new_tokens: int | None = None,
                              min_new_tokens: int = 50, slot_base: int = 0) -> list:
        """Hot path only: prompt ids (host) -> waveforms (host).  Used by bench.py's end-to-end leg.
        ``slot_base`` offsets the sampler's Philox slot index so chunks / ranks under one seed draw independently."""
        gen = self._generate_ids(prompts, max_new_tokens, min_new_tokens, slot_base)
        return [self._watermark(w) for w in self._decode_codes([self._ids_to_codes(g) for g in gen])]

    def infer_batch(self, texts: Sequence[str], ref_codes: Sequence, ref_texts: Sequence[str], distributed: bool = False) -> list:
        """List in / list out.  With ``distributed=True`` (inside an initialised torch.distributed job) the
        utterances are sharded over ranks and every rank returns all waveforms (one all-gather)."""
        if not (len(texts) == len(ref_codes) == len(ref_texts)):
            raise ValueError("texts, ref_codes and ref_texts must have the same length")
        prompts = [self._apply_chat_template(c, rt, t) for t, c, rt in zip(texts, ref_codes, ref_texts)]
        if not distributed:
            out = []
            for j in range(0, len(prompts), self.max_batch):
                out += self.infer_from_prompt_ids(prompts[j: j + self.max_batch], slot_base=j)
            return out
        from neutts_air_b200 import dist

        mine = dist.shard_indices(len(prompts), [len(p) for p in prompts])
        local = []
        rank = dist.world()[0]
        for j in range(0, len(mine), self.max_batch):
            local += self.infer_from_prompt_ids([prompts[i] for i in mine[j: j + self.max_batch]], slot_base=(rank << 20) + j)
        return dist.all_gather_waveforms(local, mine, len(prompts), device=self.codec.device)

    def infer_stream(self, text: str, ref_codes, ref_text: str) -> Generator[np.ndarray, None, None]:
        """Streaming synthesis with the reference's window geometry (``neutts/neutts.py:373-465``):
        every 25 new frames (once 5 look-ahead frames exist) the codec re-decodes
        [n - 50 - 1, n + 25 + 5 + 1) and the chunk is cross-faded with triangular weights."""
        if self._is_quantized_model:  # kept for signature parity; never true on this build
            raise NotImplementedError("GGUF streaming is not part of the B200 build")
        prompt = self._apply_chat_template(ref_codes, ref_text, text)
        return self._stream(prompt, [int(c) for c in (ref_codes.tolist() if hasattr(ref_codes, "tolist") else ref_codes)])

    def infer_stream_batch(self, texts: Sequence[str], ref_codes: Sequence, ref_texts: Sequence[str]) -> Generator[list, None, None]:
        """Streaming synthesis of up to ``max_batch`` utterances at once (BASELINE.json configs[4]; the reference
        streams one utterance, ``neutts/neutts.py:373-465``).  Every yield is a list with one entry per utterance:
        the next audio chunk (float32, cross-faded exactly as in ``infer_stream``) or ``None`` when that utterance
        has nothing new.  The sequences decode in lock-step in ONE persistent-kernel launch per round; the windows
        that are due are gathered on the device from the code history and go through the codec as one batch."""
        if not (len(texts) == len(ref_codes) == len(ref_texts)):
            raise ValueError("texts, ref_codes and ref_texts must have the same length")
        prompts = [self._apply_chat_template(c, rt, t) for t, c, rt in zip(texts, ref_codes, ref_texts)]
        refs = [[int(c) for c in (rc.tolist() if hasattr(rc, "tolist") else rc)] for rc in ref_codes]
        return self._stream_batch(prompts, refs)

    def _stream(self, prompt, ref_codes) -> Generator[np.ndarray, None, None]:
        for out in self._stream_batch([prompt], [list(ref_codes)]):
            if out[0] is not None:
                yield out[0]

    def _stream_batch(self, prompts, refs) -> Generator[list, None, None]:
        """Window geometry of the reference (``neutts/neutts.py:87-91,401-421,443-465``): once F + LA undecoded frames
        exist, the codec decodes [n_dec - LB - OV, n_dec + F + LA) and the slice [n_dec - OV, n_dec + F + OV) is
        cross-faded at stride F * hop; a ragged tail closes the stream.  ``streaming_frames_per_chunk`` may be set to
        50 for the "codec every 50 tokens" configuration BASELINE.json names.

        State per slot: the code history (reference codes, then generated ones) lives ON THE DEVICE next to the
        engine's ``out_tokens``; a round is  decode(k steps, all slots) -> absorb the new tokens into the history
        with device ops -> one small D2H read of (n_generated, done, history length) -> batched codec call."""
        hop, F, LA, LB, OV = self.hop_length, self.streaming_frames_per_chunk, self.streaming_lookforward, \
            self.streaming_lookback, self.streaming_overlap_frames
        eos = self._tok_id("<|SPEECH_GENERATION_END|>")
        seed = self.seed if self.seed is not None else int(torch.randint(0, 2**31 - 1, (1,)).item())
        lm = self.backbone
        if not hasattr(lm, "prefill"):
            raise NotImplementedError("Streaming needs the neutts_air_b200.SpeechLM backbone")
        B = len(prompts)
        limits = [min(self.max_context - len(p), lm.max_new) for p in prompts]
        if min(limits) < 1:
            raise ValueError("prompt already at max_length")
        limit = max(limits)
        sp = lm.sampling(eos, 50, limit, 50, 1.0, seed) if min(limits) == limit else lm.sampling(eos, 50, limit, 50, 1.0, seed, limits=limits)
        dev = lm.out_tokens.device
        cap = max(len(r) for r in refs) + limit
        hist = torch.zeros(B, cap + 1, dtype=torch.long, device=dev)          # column `cap` is a scratch slot for masked writes
        for b, r in enumerate(refs):
            hist[b, : len(r)] = torch.as_tensor(r, dtype=torch.long)
        hlen = torch.tensor([len(r) for r in refs], dtype=torch.long, device=dev)
        absorbed = torch.zeros(B, dtype=torch.long, device=dev)                # generated tokens already looked at
        n_dec = [len(r) for r in refs]
        fades = [_CrossFade(self.streaming_stride_samples) for _ in range(B)]
        tail_done = [False] * B
        lim_t = torch.tensor(limits, dtype=torch.long)

        def absorb(lo: int, hi: int):
            """tokens [lo, hi) of every slot -> history (non-speech ids dropped, as the reference's regex does)"""
            if hi <= lo:
                return
            ngen = lm.n_generated[:B].long()
            seg, ok = self._ids_to_codes_masked(lm.out_tokens[:B, lo:hi].long())
            cols = torch.arange(lo, hi, device=dev)[None, :]
            valid = (cols >= absorbed[:, None]) & (cols < ngen[:, None]) & ok
            pos = hlen[:, None] + torch.cumsum(valid, 1) - 1
            hist.scatter_(1, torch.where(valid, pos, torch.full_like(pos, cap)), seg)
            hlen.add_(valid.sum(1))
            absorbed.copy_(torch.minimum(ngen, torch.full_like(ngen, hi)))

        def decode_windows(jobs):
            """jobs: (slot, t0, t1, s0, s1 | None) -> one waveform slice per job, in job order.  A codec with
            ``decode_code_ragged`` takes every window of the round in calls of at most ``max_batch``, gathered from the
            history with one flat index; any other codec gets one ``decode_code`` call per window length."""
            out = [None] * len(jobs)
            cbatch = max(1, getattr(self.codec, "max_batch", 1))
            ragged = hasattr(self.codec, "decode_code_ragged")
            if ragged:
                groups = [list(range(g0, min(g0 + cbatch, len(jobs)))) for g0 in range(0, len(jobs), cbatch)]
            else:
                by_len = {}
                for i, j in enumerate(jobs):
                    by_len.setdefault(j[2] - j[1], []).append(i)
                groups = [g[g0: g0 + cbatch] for g in by_len.values() for g0 in range(0, len(g), cbatch)]
            for g in groups:
                lens = [jobs[i][2] - jobs[i][1] for i in g]
                with torch.no_grad():
                    if ragged:
                        flat = torch.cat([torch.arange(jobs[i][0] * (cap + 1) + jobs[i][1], jobs[i][0] * (cap + 1) + jobs[i][2])
                                          for i in g])
                        codes = hist.view(-1)[flat.to(dev)]
                        wavs = _split_frames(self.codec.decode_code_ragged(codes.to(self.codec.device), lens).cpu().numpy(), lens)
                    else:
                        rows = torch.tensor([jobs[i][0] for i in g], device=dev)
                        idx = torch.tensor([jobs[i][1] for i in g], device=dev)[:, None] + torch.arange(lens[0], device=dev)[None, :]
                        codes = hist[rows[:, None], idx][:, None, :]
                        wavs = list(self.codec.decode_code(codes.to(self.codec.device))[:, 0, :].cpu().numpy())
                for i, pcm in zip(g, wavs):
                    s0, s1 = jobs[i][3], jobs[i][4]
                    wav = self._watermark(pcm)
                    out[i] = wav[max(s0, 0):] if s1 is None else wav[s0:s1]
            return out

        lm.prefill(prompts, sp)             # samples the first token of every slot
        lo, hi = 0, 1
        while True:
            absorb(lo, hi)
            st = torch.stack((lm.n_generated[:B].long(), lm.done[:B].long(), hlen)).cpu()   # the round's one D2H read
            ngen_h, done_h, hlen_h = st[0], st[1], st[2]
            finished = [bool(done_h[b]) or int(ngen_h[b]) >= limits[b] for b in range(B)]
            jobs = []
            for b in range(B):
                while int(hlen_h[b]) - n_dec[b] >= F + LA:
                    t0 = max(n_dec[b] - LB - OV, 0)
                    # the reference slices up to n_dec + F + LA + OV, but tokens arrive one at a time there, so
                    # its cache never holds more than n_dec + F + LA entries when a chunk fires (:401-415)
                    t1 = n_dec[b] + F + LA
                    s0 = (n_dec[b] - t0) * hop
                    jobs.append((b, t0, t1, s0, s0 + (F + 2 * OV) * hop))
                    n_dec[b] += F
            # ragged tail of a slot that finished (neutts/neutts.py:443-465), once its regular chunks are out; the
            # tails go through the codec together with this round's regular windows
            has_chunk = {j[0] for j in jobs}
            tails, flushes = [], []
            all_finished = all(finished)
            for b in range(B):
                if finished[b] and not tail_done[b] and (all_finished or b not in has_chunk):
                    tail_done[b] = True
                    n = int(hlen_h[b])
                    if n > n_dec[b]:
                        rem = n - n_dec[b]
                        t0 = max(n - (LB + OV + rem), 0)
                        tails.append((b, t0, n, (n - t0 - rem - OV) * hop, None))
                    else:
                        flushes.append(b)
            wavs = decode_windows(jobs + tails) if jobs or tails else []
            out = [None] * B
            for b in sorted(has_chunk):
                out[b] = np.concatenate([fades[b].push(w) for j, w in zip(jobs, wavs) if j[0] == b])
            for b in flushes:
                if fades[b].acc.shape[0]:
                    flush = fades[b].push(np.zeros(0, np.float32), final=True)
                    out[b] = flush if out[b] is None else np.concatenate((out[b], flush))
            if all_finished and any(o is not None for o in out) and tails:
                yield out                    # regular chunks first: a tail is its own yield, as in the reference
                out = [None] * B
            for (b, *_), w in zip(tails, wavs[len(jobs):]):
                t = fades[b].push(w, final=True)
                out[b] = t if out[b] is None else np.concatenate((out[b], t))
            if any(o is not None for o in out):
                yield out
            if all_finished:
                break
            # decode just enough steps for the next chunk of the most advanced unfinished slot to fire (non-speech
            # ids may make it take another pass); finished slots idle inside the kernel
            need = min(F + LA - (int(hlen_h[b]) - n_dec[b]) for b in range(B) if not finished[b])
            room = min(limits[b] - int(ngen_h[b]) for b in range(B) if not finished[b])
            steps = max(1, min(need, room))
            lo = min(int(ngen_h[b]) for b in range(B) if not finished[b])   # finished slots were absorbed completely above
            lm.decode(steps, sp)
            hi = int(ngen_h.max()) + steps

    def encode_reference(self, ref_audio_path):
        """wav -> NeuCodec codes (``neutts/neutts.py:266-271``).  The encoder is outside the hot path; this
        delegates to ``codec.encode_code`` (the real ``neucodec`` when installed) or loads pre-encoded
        ``.pt`` / ``.npy`` codes saved by ``examples/encode_reference.py``."""
        p = Path(ref_audio_path)
        if p.suffix == ".pt":
            return torch.load(p)
        if p.suffix == ".npy":
            return torch.from_numpy(np.load(p))
        try:
            import librosa

            wav, _ = librosa.load(ref_audio_path, sr=16000, mono=True)
            wav_tensor = torch.from_numpy(wav).float().unsqueeze(0).unsqueeze(0)
            with torch.no_grad():
                return self.codec.encode_code(audio_or_path=wav_tensor).squeeze(0).squeeze(0)
        except ImportError as e:
            # neither librosa nor the neucodec encoder is installed: use the pre-encoded codes that sit next to
            # the audio (the reference ships samples/dave.wav + samples/dave.pt, examples/README.md:15-23)
            for ext in (".pt", ".npy"):
                q = p.with_suffix(ext)
                if q.exists():
                    warnings.warn(f"{e}; using the pre-encoded reference codes {q.name}")
                    return torch.load(q) if ext == ".pt" else torch.from_numpy(np.load(q))
            raise ImportError(f"cannot encode {p.name}: {e} (and no pre-encoded {p.stem}.pt / .npy next to it)") from e
