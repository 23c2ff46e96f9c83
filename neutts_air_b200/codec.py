"""NeuCodec decoder engine on the C-ABI (inner seam 2 of the reference: an object with ``.device``,
``.decode_code(LongTensor[B,1,N]) -> FloatTensor[B,1,480N]``, ``.eval()``, ``.to()`` —
``neutts/neutts.py:189,288-291``)."""
from __future__ import annotations

import ctypes as C
import itertools
import math
from collections.abc import Sequence
from dataclasses import dataclass

import torch

from . import _lib


@dataclass
class CodecShape:
    """Decoder shape (defaults: NeuCodec as described in SURVEY.md §3.4; a real checkpoint's
    state_dict overrides them in ``loader.codec_shape_from_state_dict``)."""

    fsq_levels: int = 4
    fsq_dims: int = 8
    quant_dim: int = 2048
    hidden: int = 1024
    depth: int = 12
    heads: int = 16
    head_dim: int = 64
    mlp_mult: int = 4
    groups: int = 32
    embed_kernel: int = 7
    n_fft: int = 1920
    hop: int = 480
    rope_base: float = 10000.0
    rope_axis: str = "time"
    norm_eps: float = 1e-6
    mag_clip: float = 1e2


def idft_basis(n_fft: int, kpad: int) -> torch.Tensor:
    """[n_fft, kpad] matrix Bm with frames = [Re | Im] @ Bm^T: inverse real DFT (norm="backward",
    imaginary parts of DC and Nyquist ignored, like torch.fft.irfft) times the periodic Hann window."""
    nb = n_fft // 2 + 1
    m = torch.arange(n_fft, dtype=torch.float64)[:, None]
    k = torch.arange(nb, dtype=torch.float64)[None, :]
    ang = 2.0 * math.pi * m * k / n_fft
    ck = torch.full((1, nb), 2.0, dtype=torch.float64)
    ck[0, 0] = 1.0
    ck[0, -1] = 1.0
    win = torch.hann_window(n_fft, periodic=True, dtype=torch.float64)[:, None]
    out = torch.zeros(n_fft, kpad, dtype=torch.float64)
    out[:, :nb] = ck * torch.cos(ang) / n_fft * win
    out[:, nb:2 * nb] = -ck * torch.sin(ang) / n_fft * win
    return out.float()


def pack_weights(shape: CodecShape, w: dict, device) -> dict:
    """``w``: dict with the decoder tensors in PyTorch layout (see ``loader.codec_weights_from_state_dict``
    for the neucodec names).  Returns fp32 device tensors in the layouts of include/neutts_b200.h."""
    dev = torch.device(device)
    f32 = lambda t: t.to(device=dev, dtype=torch.float32).contiguous()
    flat = lambda cw: cw.permute(0, 2, 1).reshape(cw.shape[0], -1)   # [Co, Ci, k] -> [Co, k*Ci] tap-major
    # collapse fc_post_a(project_out(z)) into one affine (float64 on the host, once)
    po_w, po_b = w["project_out_w"].double(), w["project_out_b"].double()
    fa_w, fa_b = w["fc_post_a_w"].double(), w["fc_post_a_b"].double()
    out = dict(fsq_w=f32(fa_w @ po_w), fsq_b=f32(fa_w @ po_b + fa_b),
               embed_w=f32(flat(w["embed_w"])), embed_b=f32(w["embed_b"]))
    rn = list(w["prior"]) + list(w["post"])
    for key in ("n1w", "n1b", "c1b", "n2w", "n2b", "c2b"):
        out["rn_" + key] = [f32(r[key]) for r in rn]
    out["rn_c1w"] = [f32(flat(r["c1w"])) for r in rn]
    out["rn_c2w"] = [f32(flat(r["c2w"])) for r in rn]
    for key in ("att_norm", "wqkv", "wproj", "ffn_norm", "fc1", "fc2"):
        out[key] = [f32(b[key]) for b in w["blocks"]]
    out["final_ln_w"], out["final_ln_b"] = f32(w["final_ln_w"]), f32(w["final_ln_b"])
    out["head_w"], out["head_b"] = f32(w["head_w"]), f32(w["head_b"])
    kpad = (shape.n_fft + 2 + 31) // 32 * 32
    out["idft_basis"] = f32(idft_basis(shape.n_fft, kpad))
    return out


class CodecDecoder:
    PRECISIONS = {"mixed": 0, "tf32": 1, "3xtf32": 2}

    def __init__(self, shape: CodecShape, weights: dict, device="cuda", max_batch: int = 1, max_frames: int = 2048,
                 precision: str = "3xtf32"):
        """``precision`` of the tensor-core GEMMs (``nt_codec_config.precision``; fp32 storage and accumulation always):
        "3xtf32" (default) = every product as three TF32 MMAs over hi/lo operand halves, fp32-grade -- the mode that meets
        the reference's fp32 path within 1e-3 RMS even on adversarial head statistics (measured 2.3e-5 at speech level
        where plain TF32 gives 2.1e-3, tests/test_gpu_codec.py); "tf32" = single-pass TF32 (~2.7x faster codec, 3.4e-4
        on speech-level weights); "mixed" = TF32 with 3xTF32 on the ISTFT head + inverse DFT only."""
        if precision not in self.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(self.PRECISIONS)}")
        if not torch.cuda.is_available():
            raise RuntimeError("neutts_air_b200.CodecDecoder needs a CUDA device (sm_100a); there is no CPU fallback")
        if shape.rope_axis not in ("time", "head"):
            raise ValueError(f"rope_axis {shape.rope_axis!r}")
        self.L = _lib.lib()
        self.shape = shape
        self.device = torch.device(device)
        self.max_batch, self.max_frames = max_batch, max_frames
        with torch.cuda.device(self.device):
            self.w = pack_weights(shape, weights, self.device)
            cfg = _lib.CodecConfig(shape.hidden, shape.depth, shape.heads, shape.head_dim, shape.mlp_mult * shape.hidden,
                                   shape.groups, shape.embed_kernel, shape.n_fft, shape.hop, shape.fsq_levels,
                                   shape.fsq_dims, shape.norm_eps, shape.rope_base, shape.mag_clip,
                                   1 if shape.rope_axis == "time" else 0, max_batch, max_frames, self.PRECISIONS[precision])
            ws_bytes = self.L.nt_codec_workspace_bytes(C.byref(cfg))
            if ws_bytes == 0:
                _lib.check(-1)
            self.workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
            keys = ("rn_n1w", "rn_n1b", "rn_c1w", "rn_c1b", "rn_n2w", "rn_n2b", "rn_c2w", "rn_c2b",
                    "att_norm", "wqkv", "wproj", "ffn_norm", "fc1", "fc2")
            self._ptrs = {k: _lib.ptr_array(self.w[k]) for k in keys}
            p = lambda k: self.w[k].data_ptr()
            wts = _lib.CodecWeights(p("fsq_w"), p("fsq_b"), p("embed_w"), p("embed_b"),
                                    *[self._ptrs[k] for k in keys],
                                    p("final_ln_w"), p("final_ln_b"), p("head_w"), p("head_b"), p("idft_basis"))
            self.handle = C.c_void_p()
            _lib.check(self.L.nt_codec_create(C.byref(cfg), C.byref(wts), self.workspace.data_ptr(), ws_bytes,
                                              C.byref(self.handle)))

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.L.nt_codec_destroy(self.handle)
        except Exception:
            pass

    # seam-compat no-ops (neutts/neutts.py:189 calls .eval().to(device))
    def eval(self):
        return self

    def to(self, device):
        if torch.device(device).type != "cuda":
            raise ValueError("neutts_air_b200.CodecDecoder runs on CUDA (sm_100a) only")
        return self

    @torch.no_grad()
    def decode_code(self, codes: torch.Tensor, validate: bool | None = None) -> torch.Tensor:
        """codes: integer [B, 1, N] (values in [0, levels**dims)) -> float32 [B, 1, hop*N] on ``self.device``.

        Range validation needs the values on the host: it runs for CPU inputs (free) and is skipped for CUDA
        inputs unless ``validate=True`` (a min/max read-back is a device synchronisation inside the hot path;
        the kernel itself never reads out of bounds on a bad id, it decodes the id modulo the codebook)."""
        if codes.dim() != 3 or codes.shape[1] != 1:
            raise ValueError("codes must be [B, 1, N]")
        B, _, N = codes.shape
        if N < 1:
            raise ValueError("No valid speech tokens found in the output.")
        cmax = self.shape.fsq_levels ** self.shape.fsq_dims
        if validate is None:
            validate = codes.device.type == "cpu"
        if validate and (int(codes.min()) < 0 or int(codes.max()) >= cmax):
            raise ValueError(f"codec ids must be in [0, {cmax})")
        with torch.cuda.device(self.device):
            c32 = codes[:, 0, :].to(self.device, torch.int32).contiguous()
            pcm = torch.empty(B, 1, self.shape.hop * N, dtype=torch.float32, device=self.device)
            _lib.check(self.L.nt_codec_decode(self.handle, c32.data_ptr(), B, N, pcm.data_ptr(), _lib.current_stream_ptr()))
        return pcm

    @torch.no_grad()
    def decode_code_ragged(self, codes: torch.Tensor, lengths: Sequence[int], validate: bool | None = None) -> torch.Tensor:
        """Items of different lengths in one codec pass.  codes: integer [T], the items packed back to back (item b =
        codes[sum(lengths[:b]) : sum(lengths[:b+1])]) -> float32 [hop*T] on ``self.device``, item b's waveform at
        [hop*sum(lengths[:b]), hop*sum(lengths[:b+1])).  Each waveform equals ``decode_code`` of that item alone.

        Needs 1..max_batch items of 1..max_frames frames each; id validation follows ``decode_code``."""
        lengths = [int(n) for n in lengths]
        if not lengths:
            raise ValueError("decode_code_ragged needs at least one item")
        if len(lengths) > self.max_batch:
            raise ValueError(f"{len(lengths)} items exceed the codec's max_batch {self.max_batch}")
        if min(lengths) < 1:
            raise ValueError("No valid speech tokens found in the output.")
        if max(lengths) > self.max_frames:
            raise ValueError(f"an item has {max(lengths)} frames, above the codec's max_frames {self.max_frames}")
        if codes.dim() != 1 or codes.shape[0] != sum(lengths):
            raise ValueError(f"codes must be 1-D with sum(lengths) = {sum(lengths)} entries, got shape {tuple(codes.shape)}")
        cmax = self.shape.fsq_levels ** self.shape.fsq_dims
        if validate is None:
            validate = codes.device.type == "cpu"
        if validate and (int(codes.min()) < 0 or int(codes.max()) >= cmax):
            raise ValueError(f"codec ids must be in [0, {cmax})")
        cu = (C.c_int32 * (len(lengths) + 1))(0, *itertools.accumulate(lengths))
        with torch.cuda.device(self.device):
            c32 = codes.to(self.device, torch.int32).contiguous()
            pcm = torch.empty(self.shape.hop * codes.shape[0], dtype=torch.float32, device=self.device)
            _lib.check(self.L.nt_codec_decode_ragged(self.handle, c32.data_ptr(), cu, len(lengths), pcm.data_ptr(),
                                                     _lib.current_stream_ptr()))
        return pcm

    def encode_code(self, audio_or_path):
        """The encoder half (wav -> codes, ``neutts/neutts.py:266-271``) is outside the hot path (SURVEY.md §2:
        one-off per speaker, pre-encodable), so it is not reimplemented: this delegates to the real ``neucodec``
        package (lazily loaded on first use, kept on this decoder's GPU) and raises ImportError with the
        pre-encoding recipe when it is not installed."""
        if getattr(self, "_encoder", None) is None:
            try:
                from neucodec import DistillNeuCodec, NeuCodec
            except ImportError as e:
                raise ImportError(
                    "encoding reference audio needs the `neucodec` package (pip install neucodec): neutts_air_b200 "
                    "implements the NeuCodec *decoder* only. Alternatively pre-encode the reference once with "
                    "examples/encode_reference.py and pass the saved .pt codes to NeuTTS.infer / encode_reference") from e
            repo = getattr(self, "repo", None) or "neuphonic/neucodec"
            cls = DistillNeuCodec if "distill" in str(repo) else NeuCodec
            self._encoder = cls.from_pretrained(repo).eval().to(self.device)
        with torch.no_grad():
            return self._encoder.encode_code(audio_or_path=audio_or_path)
