// NeuCodec decoder (seam 2: neutts/neutts.py:288-291 -> codec.decode_code) for sm_100a.
//
// Activations are channels-last fp32 in a padded-batch layout: item b owns the N_b + 6 rows starting at
// row0_b = sum_{j<b} (N_j + 6); frame t sits at row row0_b + 3 + t and the 3 rows on either side stay zero, so every
// Conv1d (k=7 and k=3, "same" padding) is a plain TMA-fed tcgen05 GEMM over all rows whose K loop walks the taps
// (gemm_tc.cu) -- no im2col buffer, no per-item launches.  Items may have different lengths (nt_codec_decode_ragged);
// the equal-length nt_codec_decode is the case N_b = N.  Per-item geometry reaches the kernels through a small device
// table (CodecItem, one async copy per call); kernels over frames run a grid over the longest item and blocks past an
// item's length return at once.
// All dense math runs on the tensor cores as TF32 with fp32 accumulation (the <=1e-3 RMS PCM
// bar of BASELINE.json rules out bf16 operands here); norms, attention softmax, exp/sin/cos
// and the overlap-add run in fp32 on CUDA cores.
//
// Pad rows: only the Conv1d inputs x0 and x2 need zero pad rows, and they are written by fsq_embed_kernel and
// groupnorm_swish_kernel alone, which touch frame rows only; the per-call memset zeroes the rest.  The GEMMs write every
// row of their outputs, so pad rows of x1 / x3 / xn / qkv / hbuf / sp / fr carry values no frame row ever reads: every
// other stage is row-local (row norms, GEMMs without taps, spec_kernel) or reads the frame rows of its own item only
// (groupnorm, attention, overlap-add).
//
// Stage map (SURVEY.md §8a):  B1+B2 fsq_embed_kernel | B3 conv-GEMM | B4 groupnorm_swish_kernel
// + conv-GEMMs | B5 rmsnorm, GEMMs, rope, codec_attn_kernel | B6 layernorm + head GEMM +
// spec_kernel | B7 inverse-rDFT GEMM + ola_kernel.
#include <cmath>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "internal.h"

namespace nt {

// one item of a codec batch: first row of its padded block, frame count, first frame in the packed codes / PCM
struct CodecItem {
  int row0, n, frame0, pad_;
};

// ------------------------------------------------------------------ B1+B2: codes -> fc_post_a(project_out(fsq))
// grid (max N, B), 256 threads.  out row = row0_b + 3 + t.
__global__ void __launch_bounds__(256) fsq_embed_kernel(const int32_t* codes, const CodecItem* items, int C, int levels, int dims,
                                                        const float* w, const float* bias, float* out) {
  pdl_launch_dependents();
  pdl_wait();
  const int t = blockIdx.x;
  const CodecItem it = items[blockIdx.y];
  if (t >= it.n) return;
  int code = codes[it.frame0 + t];
  float z[16];
  const float half = static_cast<float>(levels / 2);
  for (int i = 0; i < dims; ++i) {
    z[i] = (static_cast<float>(code % levels) - half) / half;
    code /= levels;
  }
  float* o = out + (static_cast<long long>(it.row0) + 3 + t) * C;
  for (int c = threadIdx.x; c < C; c += 256) {
    float acc = bias[c];
    for (int i = 0; i < dims; ++i) acc += w[c * dims + i] * z[i];
    o[c] = acc;
  }
}

// ------------------------------------------------------------------ B4: GroupNorm + swish
// grid (groups, B), 256 threads.  cpg = C/groups channels (<= 32) x N_b frames per group.
__global__ void __launch_bounds__(256) groupnorm_swish_kernel(const float* x, const CodecItem* items, int C, int cpg, float eps,
                                                              const float* gw, const float* gb, float* out) {
  __shared__ float red[8];
  __shared__ float s_stat;
  pdl_launch_dependents();
  pdl_wait();
  const int g = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const CodecItem it = items[blockIdx.y];
  const int N = it.n;
  const long long base = (static_cast<long long>(it.row0) + 3) * C + g * cpg;
  const float cnt = static_cast<float>(N) * cpg;
  auto block_sum = [&](float v) {
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (tid == 0) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += red[i];
      s_stat = t;
    }
    __syncthreads();
    return s_stat;
  };
  float s = 0.f;
  if (lane < cpg)
    for (int t = warp; t < N; t += 8) s += x[base + static_cast<long long>(t) * C + lane];
  const float mean = block_sum(s) / cnt;
  float v = 0.f;
  if (lane < cpg)
    for (int t = warp; t < N; t += 8) {
      const float d = x[base + static_cast<long long>(t) * C + lane] - mean;
      v += d * d;
    }
  const float rstd = rsqrtf(block_sum(v) / cnt + eps);
  if (lane < cpg) {
    const float w = gw[g * cpg + lane], bb = gb[g * cpg + lane];
    for (int t = warp; t < N; t += 8) {
      const float y = (x[base + static_cast<long long>(t) * C + lane] - mean) * rstd * w + bb;
      out[base + static_cast<long long>(t) * C + lane] = y / (1.0f + __expf(-y));
    }
  }
}

// ------------------------------------------------------------------ row norms (one warp per row, all rows)
// mode 0: RMSNorm (x * rsqrt(mean x^2 + eps) * w); mode 1: LayerNorm with bias
__global__ void __launch_bounds__(256) rownorm_kernel(const float* x, int rows, int C, float eps, const float* w,
                                                      const float* bias, int mode, float* out) {
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + static_cast<long long>(row) * C;
  float* orow = out + static_cast<long long>(row) * C;
  float mean = 0.f;
  if (mode == 1) {
    float s = 0.f;
    for (int i = lane; i < C; i += 32) s += xr[i];
    mean = warp_sum(s) / static_cast<float>(C);
  }
  float v = 0.f;
  for (int i = lane; i < C; i += 32) {
    const float d = xr[i] - mean;
    v += d * d;
  }
  const float rstd = rsqrtf(warp_sum(v) / static_cast<float>(C) + eps);
  for (int i = lane; i < C; i += 32) {
    float y = (xr[i] - mean) * rstd * w[i];
    if (mode == 1) y += bias[i];
    orow[i] = y;
  }
}

// ------------------------------------------------------------------ B5: rotary on q,k (interleaved pairs, frame index)
// grid (max N, B), threads = heads*32 pairs; t restarts at 0 in every item.  qkv row layout: [q(h,d) | k(h,d) | v(h,d)]
__global__ void codec_rope_kernel(float* qkv, const CodecItem* items, int C, int heads, const float* inv_freq) {
  pdl_launch_dependents();
  pdl_wait();
  const int t = blockIdx.x;
  const CodecItem it = items[blockIdx.y];
  if (t >= it.n) return;
  float* row = qkv + (static_cast<long long>(it.row0) + 3 + t) * 3 * C;
  for (int i = threadIdx.x; i < heads * 32; i += blockDim.x) {
    const int h = i >> 5, pr = i & 31;
    float s, c;
    sincosf(static_cast<float>(t) * inv_freq[pr], &s, &c);
#pragma unroll
    for (int which = 0; which < 2; ++which) {
      float2* p = reinterpret_cast<float2*>(row + which * C + h * 64 + 2 * pr);
      const float2 v = *p;
      *p = make_float2(v.x * c - v.y * s, v.y * c + v.x * s);
    }
  }
}

// ------------------------------------------------------------------ B5: bidirectional attention, fp32
// grid (ceil(max N/128), heads, B), 128 threads; thread = one query row; K/V tiles of 32 frames in smem.
// Blocks past the item's length return before the first __syncthreads (the exit is block-uniform).
__global__ void __launch_bounds__(128) codec_attn_kernel(const float* qkv, const CodecItem* items, int C, float scale_log2, float* out) {
  __shared__ __align__(16) float sK[32 * 64];
  __shared__ __align__(16) float sV[32 * 64];
  pdl_launch_dependents();
  pdl_wait();
  const int qb = blockIdx.x, h = blockIdx.y, tid = threadIdx.x;
  const CodecItem it = items[blockIdx.z];
  const int N = it.n;
  if (qb * 128 >= N) return;
  const int tq = qb * 128 + tid;
  const bool active = tq < N;
  const long long row0 = static_cast<long long>(it.row0) + 3;
  float q[64], o[64], m = -INFINITY, l = 0.f;
  if (active) {
    const float4* qp = reinterpret_cast<const float4*>(qkv + (row0 + tq) * 3 * C + h * 64);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float4 v = qp[j];
      q[4 * j] = v.x * scale_log2, q[4 * j + 1] = v.y * scale_log2, q[4 * j + 2] = v.z * scale_log2, q[4 * j + 3] = v.w * scale_log2;
    }
  }
#pragma unroll
  for (int j = 0; j < 64; ++j) o[j] = 0.f;
  const int ntiles = (N + 31) >> 5;
  for (int tile = 0; tile < ntiles; ++tile) {
    const int k0 = tile * 32;
    __syncthreads();
    for (int i = tid; i < 32 * 16; i += 128) {
      const int j = i >> 4, c4 = i & 15;
      float4 kv4 = make_float4(0.f, 0.f, 0.f, 0.f), vv4 = kv4;
      if (k0 + j < N) {
        const float* r = qkv + (row0 + k0 + j) * 3 * C + h * 64;
        kv4 = reinterpret_cast<const float4*>(r + C)[c4];
        vv4 = reinterpret_cast<const float4*>(r + 2 * C)[c4];
      }
      reinterpret_cast<float4*>(sK)[i] = kv4;
      reinterpret_cast<float4*>(sV)[i] = vv4;
    }
    __syncthreads();
    if (!active) continue;
    float s[32], tmax = -INFINITY;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      float d = 0.f;
      const float4* kr = reinterpret_cast<const float4*>(sK + j * 64);
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        const float4 f = kr[c];
        d += q[4 * c] * f.x + q[4 * c + 1] * f.y + q[4 * c + 2] * f.z + q[4 * c + 3] * f.w;
      }
      s[j] = (k0 + j < N) ? d : -INFINITY;
      tmax = fmaxf(tmax, s[j]);
    }
    const float mn = fmaxf(m, tmax);
    const float corr = exp2f(m - mn);
    l *= corr;
#pragma unroll
    for (int j = 0; j < 64; ++j) o[j] *= corr;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float pj = exp2f(s[j] - mn);
      l += pj;
      const float4* vr = reinterpret_cast<const float4*>(sV + j * 64);
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        const float4 f = vr[c];
        o[4 * c] += pj * f.x, o[4 * c + 1] += pj * f.y, o[4 * c + 2] += pj * f.z, o[4 * c + 3] += pj * f.w;
      }
    }
    m = mn;
  }
  if (active) {
    const float inv = 1.0f / l;
    float4* op = reinterpret_cast<float4*>(out + (row0 + tq) * C + h * 64);
#pragma unroll
    for (int j = 0; j < 16; ++j) op[j] = make_float4(o[4 * j] * inv, o[4 * j + 1] * inv, o[4 * j + 2] * inv, o[4 * j + 3] * inv);
  }
}

// ------------------------------------------------------------------ B6: (log-mag | phase) -> (Re | Im), in place
// sp row layout: [nb log-magnitudes][nb phases][pad];  grid rows, 256 threads
__global__ void spec_kernel(float* sp, long long ld, int nb, float clip) {
  pdl_launch_dependents();
  pdl_wait();
  float* r = sp + blockIdx.x * ld;
  for (int k = threadIdx.x; k < nb; k += blockDim.x) {
    const float mag = fminf(expf(r[k]), clip);
    float s, c;
    sincosf(r[nb + k], &s, &c);
    r[k] = mag * c;
    r[nb + k] = mag * s;
  }
}

// ------------------------------------------------------------------ B7: overlap-add + envelope ("same" padding)
// frames rows already carry the synthesis window (folded into the inverse-rDFT basis).
// grid (ceil(hop * max N / 256), B); item b's hop*N_b samples start at pcm[hop * frame0_b].
__global__ void __launch_bounds__(256) ola_kernel(const float* frames, const CodecItem* items, int n_fft, int hop, float* pcm) {
  pdl_launch_dependents();
  pdl_wait();
  const CodecItem it = items[blockIdx.y];
  const int N = it.n;
  const int n = blockIdx.x * 256 + threadIdx.x;
  const int total = hop * N;
  if (n >= total) return;
  const int pad = (n_fft - hop) / 2;
  const int np = n + pad;  // index in the un-trimmed signal
  int t_hi = np / hop;
  if (t_hi > N - 1) t_hi = N - 1;
  float acc = 0.f, env = 0.f;
  const float w0 = 6.283185307179586f / static_cast<float>(n_fft);
  for (int t = t_hi; t >= 0; --t) {
    const int m = np - t * hop;
    if (m >= n_fft) break;
    acc += frames[(static_cast<long long>(it.row0) + 3 + t) * n_fft + m];
    const float w = 0.5f * (1.0f - cosf(w0 * static_cast<float>(m)));
    env += w * w;
  }
  pcm[static_cast<long long>(hop) * it.frame0 + n] = acc / env;
}

// 3xTF32 operand split: hi = x rounded to the 10-bit TF32 mantissa (exactly representable, so the tensor core's own
// fp32 -> tf32 conversion leaves it alone), lo = x - hi (exact in fp32).  A.W ~ A_lo.W_hi + A_hi.W_lo + A_hi.W_hi with
// fp32 accumulation is accurate to ~2^-21 per product instead of 2^-11.
__global__ void split_tf32_kernel(const float* __restrict__ x, float* __restrict__ hi, float* __restrict__ lo, long long n) {
  pdl_launch_dependents();
  pdl_wait();
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float v = x[i];
    const float h = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
    hi[i] = h;
    lo[i] = v - h;
  }
}

}  // namespace nt

using namespace nt;

struct SplitW {   // hi / lo halves of one weight matrix (workspace: lo directly below hi, `rows` rows further down);
  float* hi = nullptr;   // null when the matrix runs in plain TF32
  float* lo = nullptr;
  int rows = 0;
};

struct nt_codec {
  nt_codec_config cfg;
  nt_codec_weights w;
  std::vector<const float*> rn[8], blk[6];
  float *x0, *x1, *x2, *x3, *xn, *qkv, *hbuf, *att, *sp, *fr, *inv_freq;
  CodecItem* items;   // [max_batch] geometry of the current call's items (filled by one async copy per call)
  int kpad;
  // 3xTF32 (cfg.precision != 1): split weights, split-activation scratch, partial-sum scratch
  SplitW s_head, s_idft, s_embed;
  std::vector<SplitW> s_rn[2], s_blk[4];   // resnet conv1 / conv2; wqkv, wproj, fc1, fc2
  float* a_split = nullptr;   // hi half, then the lo half a_rows rows further down (placed per GEMM)
};

static int codec_check(const nt_codec_config* c) {
  if (!c) return set_error(NT_ERR_INVALID, "null codec config");
  if (c->head_dim != 64 || c->heads * 64 != c->hidden) return set_error(NT_ERR_INVALID, "codec: heads*64 must equal hidden");
  if (c->hidden % 32 || c->mlp_hidden % 32) return set_error(NT_ERR_INVALID, "codec: hidden sizes must be multiples of 32");
  if (c->groups < 1 || c->hidden % c->groups || c->hidden / c->groups > 32) return set_error(NT_ERR_INVALID, "codec: unsupported group count");
  if (c->embed_kernel != 7) return set_error(NT_ERR_INVALID, "codec: embed kernel must be 7");
  if (c->fsq_dims > 16 || c->fsq_levels < 2) return set_error(NT_ERR_INVALID, "codec: unsupported FSQ shape");
  if (c->n_fft % 4 || c->hop < 1 || (c->n_fft - c->hop) % 2 || c->n_fft < c->hop) return set_error(NT_ERR_INVALID, "codec: unsupported STFT geometry");
  if (c->max_batch < 1 || c->max_frames < 1) return set_error(NT_ERR_INVALID, "codec: bad sizes");
  if (c->precision < 0 || c->precision > 2) return set_error(NT_ERR_INVALID, "codec: precision %d not in 0..2", c->precision);
  return NT_OK;
}

static size_t codec_carve(const nt_codec_config& c, void* ws, size_t bytes, nt_codec* k) {
  Arena a(ws, bytes);
  const size_t rows = size_t(c.max_batch) * (c.max_frames + 6) + 8;
  const int kpad = ((c.n_fft + 2 + 31) / 32) * 32;
  k->kpad = kpad;
  k->x0 = a.take<float>(rows * c.hidden);
  k->x1 = a.take<float>(rows * c.hidden);
  k->x2 = a.take<float>(rows * c.hidden);
  k->x3 = a.take<float>(rows * c.hidden);
  k->xn = a.take<float>(rows * c.hidden);
  k->qkv = a.take<float>(rows * 3 * c.hidden);
  k->hbuf = a.take<float>(rows * c.mlp_hidden);
  k->att = a.take<float>(rows * c.hidden);
  k->sp = a.take<float>(rows * kpad);
  k->fr = a.take<float>(rows * c.n_fft);
  k->inv_freq = a.take<float>(64);
  k->items = a.take<CodecItem>(c.max_batch);
  if (c.precision != 1) {
    const size_t C = c.hidden, nb2 = size_t(c.n_fft) + 2;
    auto takew = [&](SplitW& w, size_t rows_, size_t ld) {   // one block: hi rows, then lo rows
      w.hi = a.take<float>(2 * rows_ * ld);
      w.lo = w.hi + rows_ * ld;
      w.rows = int(rows_);
    };
    takew(k->s_head, nb2, C);
    takew(k->s_idft, size_t(c.n_fft), kpad);
    size_t widest = kpad > c.n_fft ? kpad : c.n_fft;
    if (c.precision == 2) {
      takew(k->s_embed, C, c.embed_kernel * C);
      for (int i = 0; i < 2; ++i) {
        k->s_rn[i].assign(4, SplitW());
        for (int j = 0; j < 4; ++j) takew(k->s_rn[i][j], C, 3 * C);
      }
      const size_t br[4] = {3 * C, C, size_t(c.mlp_hidden), C}, bl[4] = {C, C, C, size_t(c.mlp_hidden)};
      for (int i = 0; i < 4; ++i) {
        k->s_blk[i].assign(c.depth, SplitW());
        for (int j = 0; j < c.depth; ++j) takew(k->s_blk[i][j], br[i], bl[i]);
      }
      if (size_t(c.mlp_hidden) > widest) widest = c.mlp_hidden;
      if (3 * C > widest) widest = 3 * C;
    }
    if (C > widest) widest = C;
    k->a_split = a.take<float>(2 * rows * widest);
  }
  return a.off;
}

extern "C" size_t nt_codec_workspace_bytes(const nt_codec_config* cfg) {
  if (codec_check(cfg)) return 0;
  nt_codec tmp;
  return codec_carve(*cfg, nullptr, 0, &tmp) + 256;
}

extern "C" int nt_codec_create(const nt_codec_config* cfg, const nt_codec_weights* w, void* workspace, size_t workspace_bytes,
                               nt_codec** out) {
  int rc = codec_check(cfg);
  if (rc) return rc;
  if (!w || !workspace || !out) return set_error(NT_ERR_INVALID, "nt_codec_create: null argument");
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return set_error(NT_ERR_INVALID, "workspace must be 256-byte aligned");
  nt_codec* k = new nt_codec();
  k->cfg = *cfg;
  k->w = *w;
  const size_t need = codec_carve(*cfg, workspace, workspace_bytes, k);
  if (need > workspace_bytes) {
    delete k;
    return set_error(NT_ERR_NOMEM, "codec workspace too small: need %zu, got %zu", need, workspace_bytes);
  }
  const float* const* rsrc[8] = {w->rn_n1w, w->rn_n1b, w->rn_c1w, w->rn_c1b, w->rn_n2w, w->rn_n2b, w->rn_c2w, w->rn_c2b};
  for (int i = 0; i < 8; ++i)
    for (int j = 0; j < 4; ++j) k->rn[i].push_back(rsrc[i][j]);
  const float* const* bsrc[6] = {w->att_norm, w->wqkv, w->wproj, w->ffn_norm, w->fc1, w->fc2};
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j < cfg->depth; ++j) k->blk[i].push_back(bsrc[i][j]);
  int dev = 0;
  cudaDeviceProp prop;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess || prop.major != 10) {
    delete k;
    return set_error(NT_ERR_CUDA, "no sm_100 CUDA device: this library has no CPU fallback");
  }
  float invf[64] = {0};
  for (int i = 0; i < 32; ++i) invf[i] = static_cast<float>(1.0 / std::pow(static_cast<double>(cfg->rope_base), (2.0 * i) / 64.0));
  if (cudaMemcpy(k->inv_freq, invf, sizeof(invf), cudaMemcpyHostToDevice) != cudaSuccess) {
    delete k;
    return set_error(NT_ERR_CUDA, "codec workspace initialisation failed");
  }
  if (cfg->precision != 1) {   // split the weights of the 3xTF32 GEMMs once
    const size_t C = cfg->hidden;
    auto splitw = [&](const float* src, const SplitW& w, size_t n) {
      if (w.hi) split_tf32_kernel<<<592, 256>>>(src, w.hi, w.lo, static_cast<long long>(n));
    };
    splitw(w->head_w, k->s_head, (size_t(cfg->n_fft) + 2) * C);
    splitw(w->idft_basis, k->s_idft, size_t(cfg->n_fft) * k->kpad);
    if (cfg->precision == 2) {
      splitw(w->embed_w, k->s_embed, C * cfg->embed_kernel * C);
      for (int j = 0; j < 4; ++j) splitw(k->rn[2][j], k->s_rn[0][j], C * 3 * C), splitw(k->rn[6][j], k->s_rn[1][j], C * 3 * C);
      const size_t bn[4] = {3 * C * C, C * C, size_t(cfg->mlp_hidden) * C, C * size_t(cfg->mlp_hidden)};
      const int bi[4] = {1, 2, 4, 5};
      for (int i = 0; i < 4; ++i)
        for (int j = 0; j < cfg->depth; ++j) splitw(k->blk[bi[i]][j], k->s_blk[i][j], bn[i]);
    }
    if (cudaDeviceSynchronize() != cudaSuccess || cudaGetLastError() != cudaSuccess) {
      delete k;
      return set_error(NT_ERR_CUDA, "codec: weight split failed");
    }
  }
  *out = k;
  return NT_OK;
}

extern "C" int nt_codec_destroy(nt_codec* c) {
  delete c;
  return NT_OK;
}

namespace {
struct CodecRun {
  nt_codec* k;
  int B, maxN, rows, C;
  cudaStream_t s;

  // GEMM on the padded layout.  masked (Conv1d and residual GEMMs): out rows r+3 for r in [0, rows-6), so the tap
  // window of every output row stays inside the buffer; A points at the first row the window of output row 0 touches.
  // Rows outside the items' frames are written too and never read (see the header comment).
  // sw (optional): the weight's hi / lo halves -> 3xTF32 in one pass of the GEMM kernel (A_lo.W_hi + A_hi.W_lo +
  // A_hi.W_hi into one TMEM accumulator); the activations are split into a hi / lo pair of buffers first.
  int gemm(const float* A, int K, int lda, const float* W, const float* bias, const float* residual, nt_act act, float* out,
           int ldc, int Nout, bool masked, const SplitW* sw = nullptr, int ldw = 0) {
    nt_gemm_args a;
    memset(&a, 0, sizeof(a));
    a.dtype = NT_TF32;
    a.M = masked ? rows - 6 : rows;
    a.N = Nout, a.K = K, a.A = A, a.lda = lda, a.W = W, a.ldw = ldw ? ldw : K;
    a.bias = bias, a.residual = residual, a.ldr = ldc, a.act = act, a.out_f32 = out, a.ldc = ldc;
    if (!sw || !sw->hi) return gemm_dispatch(a, s, nullptr, true);
    const int a_rows = a.M + (K + lda - 1) / lda - 1;                      // rows the tap window touches
    const long long a_elems = static_cast<long long>(a_rows) * lda;
    float* a_hi = k->a_split;
    int rc = launch_kernel(split_tf32_kernel, dim3(296), dim3(256), 0, s, true, A, a_hi, a_hi + a_elems, a_elems);
    if (rc) return rc;
    a.A = a_hi, a.W = sw->hi;
    const Split3 s3{a_rows, sw->rows};
    return gemm_dispatch(a, s, nullptr, true, &s3);
  }
  const SplitW* sp(const std::vector<SplitW>& v, int i) const { return v.empty() ? nullptr : &v[i]; }
  int resnet(int idx) {
    const nt_codec_config& c = k->cfg;
    const int cpg = C / c.groups;
    int rc;
    if ((rc = launch_kernel(groupnorm_swish_kernel, dim3(c.groups, B), dim3(256), 0, s, true, (const float*)k->x1,
                            (const CodecItem*)k->items, C, cpg, c.norm_eps, k->rn[0][idx], k->rn[1][idx], k->x2)))
      return rc;
    if ((rc = gemm(k->x2 + 2 * C, 3 * C, C, k->rn[2][idx], k->rn[3][idx], nullptr, NT_ACT_NONE, k->x3 + 3 * C, C, C, true, sp(k->s_rn[0], idx))))
      return rc;
    if ((rc = launch_kernel(groupnorm_swish_kernel, dim3(c.groups, B), dim3(256), 0, s, true, (const float*)k->x3,
                            (const CodecItem*)k->items, C, cpg, c.norm_eps, k->rn[4][idx], k->rn[5][idx], k->x2)))
      return rc;
    return gemm(k->x2 + 2 * C, 3 * C, C, k->rn[6][idx], k->rn[7][idx], k->x1 + 3 * C, NT_ACT_NONE, k->x1 + 3 * C, C, C, true, sp(k->s_rn[1], idx));
  }
};

// One forward pass over B items with frame counts cu_frames[b+1] - cu_frames[b] (host, already validated).
int codec_forward(nt_codec* k, const int32_t* codes, const int32_t* cu_frames, int B, float* pcm, cudaStream_t s) {
  const nt_codec_config& c = k->cfg;
  std::vector<CodecItem> items(B);
  int rows = 0, maxN = 0;
  for (int b = 0; b < B; ++b) {
    const int n = cu_frames[b + 1] - cu_frames[b];
    items[b] = CodecItem{rows, n, cu_frames[b], 0};
    rows += n + 6;
    if (n > maxN) maxN = n;
  }
  const int C = c.hidden;
  CodecRun r{k, B, maxN, rows, C, s};
  int rc;
  // the host vector is pageable: the runtime stages it before returning, so it may go out of scope
  NT_CUDA_CHECK(cudaMemcpyAsync(k->items, items.data(), B * sizeof(CodecItem), cudaMemcpyHostToDevice, s));
  const CodecItem* it = k->items;
  const size_t act_bytes = size_t(rows + 8) * C * sizeof(float);
  NT_CUDA_CHECK(cudaMemsetAsync(k->x0, 0, act_bytes, s));
  NT_CUDA_CHECK(cudaMemsetAsync(k->x1, 0, act_bytes, s));
  NT_CUDA_CHECK(cudaMemsetAsync(k->x2, 0, act_bytes, s));

  // B1+B2
  if ((rc = launch_kernel(fsq_embed_kernel, dim3(maxN, B), dim3(256), 0, s, true, codes, it, C, c.fsq_levels, c.fsq_dims,
                          k->w.fsq_w, k->w.fsq_b, k->x0)))
    return rc;
  // B3: Conv1d k=7 pad=3
  if ((rc = r.gemm(k->x0, 7 * C, C, k->w.embed_w, k->w.embed_b, nullptr, NT_ACT_NONE, k->x1 + 3 * C, C, C, true, &k->s_embed))) return rc;
  // B4: prior_net
  for (int i = 0; i < 2; ++i)
    if ((rc = r.resnet(i))) return rc;
  // B5: transformer blocks
  const float scale_log2 = 0.125f * 1.4426950408889634f;
  for (int l = 0; l < c.depth; ++l) {
    if ((rc = launch_kernel(rownorm_kernel, dim3((rows + 7) / 8), dim3(256), 0, s, true, (const float*)k->x1, rows, C, c.norm_eps,
                            k->blk[0][l], (const float*)nullptr, 0, k->xn)))
      return rc;
    if ((rc = r.gemm(k->xn, C, C, k->blk[1][l], nullptr, nullptr, NT_ACT_NONE, k->qkv, 3 * C, 3 * C, false, r.sp(k->s_blk[0], l)))) return rc;
    if (c.rope_time_axis)
      if ((rc = launch_kernel(codec_rope_kernel, dim3(maxN, B), dim3(256), 0, s, true, k->qkv, it, C, c.heads, (const float*)k->inv_freq)))
        return rc;
    if ((rc = launch_kernel(codec_attn_kernel, dim3((maxN + 127) / 128, c.heads, B), dim3(128), 0, s, true, (const float*)k->qkv, it, C,
                            scale_log2, k->att)))
      return rc;
    if ((rc = r.gemm(k->att + 3 * C, C, C, k->blk[2][l], nullptr, k->x1 + 3 * C, NT_ACT_NONE, k->x1 + 3 * C, C, C, true, r.sp(k->s_blk[1], l))))
      return rc;
    if ((rc = launch_kernel(rownorm_kernel, dim3((rows + 7) / 8), dim3(256), 0, s, true, (const float*)k->x1, rows, C, c.norm_eps,
                            k->blk[3][l], (const float*)nullptr, 0, k->xn)))
      return rc;
    if ((rc = r.gemm(k->xn, C, C, k->blk[4][l], nullptr, nullptr, NT_ACT_SILU, k->hbuf, c.mlp_hidden, c.mlp_hidden, false, r.sp(k->s_blk[2], l))))
      return rc;
    if ((rc = r.gemm(k->hbuf + 3 * size_t(c.mlp_hidden), c.mlp_hidden, c.mlp_hidden, k->blk[5][l], nullptr, k->x1 + 3 * C, NT_ACT_NONE,
                     k->x1 + 3 * C, C, C, true, r.sp(k->s_blk[3], l))))
      return rc;
  }
  // post_net
  for (int i = 2; i < 4; ++i)
    if ((rc = r.resnet(i))) return rc;
  // B6: final LayerNorm, head, spectrum
  if ((rc = launch_kernel(rownorm_kernel, dim3((rows + 7) / 8), dim3(256), 0, s, true, (const float*)k->x1, rows, C, c.norm_eps,
                          k->w.final_ln_w, k->w.final_ln_b, 1, k->xn)))
    return rc;
  const int nb = c.n_fft / 2 + 1, kp = k->kpad;
  if ((rc = r.gemm(k->xn, C, C, k->w.head_w, k->w.head_b, nullptr, NT_ACT_NONE, k->sp, kp, 2 * nb, false, &k->s_head))) return rc;
  if ((rc = launch_kernel(spec_kernel, dim3(rows), dim3(256), 0, s, true, k->sp, (long long)kp, nb, c.mag_clip))) return rc;
  // B7: inverse rDFT (windowed basis) as a GEMM, then overlap-add
  if ((rc = r.gemm(k->sp, 2 * nb, kp, k->w.idft_basis, nullptr, nullptr, NT_ACT_NONE, k->fr, c.n_fft, c.n_fft, false, &k->s_idft, kp))) return rc;
  return launch_kernel(ola_kernel, dim3((c.hop * maxN + 255) / 256, B), dim3(256), 0, s, true, (const float*)k->fr, it, c.n_fft, c.hop, pcm);
}
}  // namespace

extern "C" int nt_codec_decode(nt_codec* k, const int32_t* codes, int B, int N, float* pcm, void* stream_) {
  if (!k || !codes || !pcm) return set_error(NT_ERR_INVALID, "nt_codec_decode: null argument");
  const nt_codec_config& c = k->cfg;
  if (B < 1 || B > c.max_batch) return set_error(NT_ERR_INVALID, "codec batch %d not in 1..%d", B, c.max_batch);
  if (N < 1 || N > c.max_frames) return set_error(NT_ERR_INVALID, "codec frames %d not in 1..%d", N, c.max_frames);
  std::vector<int32_t> cu(B + 1);
  for (int b = 0; b <= B; ++b) cu[b] = b * N;
  return codec_forward(k, codes, cu.data(), B, pcm, reinterpret_cast<cudaStream_t>(stream_));
}

extern "C" int nt_codec_decode_ragged(nt_codec* k, const int32_t* codes, const int32_t* cu_frames, int B, float* pcm, void* stream_) {
  if (!k || !codes || !cu_frames || !pcm) return set_error(NT_ERR_INVALID, "nt_codec_decode_ragged: null argument");
  const nt_codec_config& c = k->cfg;
  if (B < 1 || B > c.max_batch) return set_error(NT_ERR_INVALID, "codec batch %d not in 1..%d", B, c.max_batch);
  if (cu_frames[0] != 0) return set_error(NT_ERR_INVALID, "codec cu_frames[0] is %d, must be 0", cu_frames[0]);
  for (int b = 0; b < B; ++b) {
    const long long n = static_cast<long long>(cu_frames[b + 1]) - cu_frames[b];
    if (n < 1 || n > c.max_frames) return set_error(NT_ERR_INVALID, "codec item %d has %lld frames, not in 1..%d", b, n, c.max_frames);
  }
  return codec_forward(k, codes, cu_frames, B, pcm, reinterpret_cast<cudaStream_t>(stream_));
}
