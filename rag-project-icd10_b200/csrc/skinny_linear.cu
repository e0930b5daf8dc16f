// skinny_linear.cu -- the encoder's linear layers for a handful of tokens (M <= 64): batch-1 encode_query.
//
// Replaces the same nn.Linear calls as gemm_tc.cu (reference call sites services/embedding_service.py:81,120 --
// model.encode of ONE text, the reference's only live usage: multi_diagnosis_service.py:152-153) when the whole batch is
// at most 64 tokens.  There the 256 x 256 tcgen05 tile is the wrong tool: a forward is 48 GEMM launches of ~11 us each
// whatever the length (r02o: 0.70 ms device-side for 12 tokens), because 3 .. 12 CTA pairs walk all of K serially and
// pull every weight through a handful of SMs (FFN-down: 3 pairs x 48 K blocks).  With so few rows the layer is a
// weight STREAM (14 MB per layer, read once) in front of a dependency wait, so this kernel is built around that:
//
//   * a warp owns EIGHT output features and a K range of 256 elements, and holds that whole 8 x 256 slice of W in
//     registers (32 per thread), loaded BEFORE griddepcontrol.wait: weights are constants, so under programmatic
//     dependent launch they stream in while the previous kernel is still finishing, and what is left after the wait
//     is a few dozen L1 / L2 reads of activation rows and the same number of MMAs;
//   * mma.sync m16n8k16 (bf16 x bf16 -> fp32; 16 tokens x 8 features): for 12 tokens there is nothing a 128-row
//     tcgen05 tile could add -- the launch is bound by latency, not by tensor throughput.  Both operands come straight
//     from global memory as 16-byte pieces: lane (r, q) reads elements [8 q, 8 q + 8) of a 32-element K block of
//     row r and uses them as the fragment pairs of TWO MMAs; the K order inside a block is permuted the same way for A
//     and W, which a dot product does not see.  (A first version on fp32 FMAs cost 16 us per token and forward: r02y.)
//   * the K / 256 warps of a feature group (3, or 12 for FFN-down) meet in shared memory and are added in a fixed order
//     (deterministic).  Short K ranges per warp are what keeps the activation loads deep: with 768 elements per warp
//     the weight slice took 96 registers, the compiler kept 8 loads in flight, and since L1 holds sectors, not lines
//     (ncu r02ah: 1.5 % L1 hits in the K-split kernels, prefetch.global.L1 notwithstanding) every 16-token tile cost
//     six L2 round trips -- 3.7 us per tile and launch;
//   * epilogue per (token, feature) as in gemm_tc.cu: bias, deferred-LayerNorm input correction, erf-GELU, residual
//     through LayerNorm.  The row statistics the deferred LayerNorm needs are computed HERE from the rows themselves
//     (<= 64 rows of H), so this path neither reads nor writes the statistics buffers of the tile kernels.
//
// The hidden size H (768 or 1024) is a template parameter: it is the row length of those statistics, the output width
// from which a layer counts as wide (4 feature groups per CTA) and it sets the warp budget of a CTA (12 / 16 warps).
// Grid per 32 tokens at 768: QKV 72 CTAs x 12 warps (4 feature groups x 3 K ranges), FFN-up 96 x 12, O 96 x 3, FFN-down
// 96 x 12; at most 16 tokens: 4 warps per CTA with 768 elements of K each (launch_skinny_linear).  At 1024: QKV 96 x 16,
// FFN-up 128 x 16, O 128 x 4, FFN-down 128 x 16; at most 16 tokens 512 elements of K per warp (8 warps; O keeps 256), since
// a 1024-element slice would be 128 registers of weights per lane (DESIGN.md).
// Roofline: latency (a few microseconds per launch); the weight stream itself is ~2 us per layer at HBM speed.
#include "common.cuh"
#include "encoder_kernels.h"
#include "ptx.cuh"

namespace icd {
namespace {

constexpr int kMaxTokens = 64;   // rows per launch (two passes of 32)
constexpr int kBlk = 8;           // 32-element K blocks per warp: a K range of 256
// 32-element K blocks per warp when the batch is one 16-token tile (the weight slice a lane keeps in registers)
constexpr int one_tile_blocks(int H) { return H == 768 ? 24 : 16; }
// warps per CTA of a kernel (its launch bound): at 768 12 for every K range; at 1024 K / 256 ranges x 4 feature groups of
// the QKV / FFN-up layers = 16 with ranges of 256 (128 registers a thread), 8 with the one-tile ranges of 512, whose
// 64 registers of weights need the larger budget of a 256-thread CTA
constexpr int max_warps(int H, int nblk) { return H == 768 ? 12 : (nblk == kBlk ? 16 : 8); }

struct SkinnyParams {
  const __nv_bfloat16* A;    // [M, K]
  const __nv_bfloat16* W;    // [N, K]
  const float* bias;         // [N]
  const float* vec2;         // [N]: c (LNIN) or gamma (residual through LayerNorm); null = neither
  const __nv_bfloat16* res;  // [M, N] residual stream or null
  __nv_bfloat16* out;        // [M, N]
  int M, N, K;
  int ks, fw;                // K splits and feature groups (of 8) per CTA: blockDim = 32 * ks * fw
  float eps;
};

__device__ __forceinline__ void unpack8(const uint4 v, float* x) {
  x[0] = bf16lo_to_f32(v.x), x[1] = bf16hi_to_f32(v.x);
  x[2] = bf16lo_to_f32(v.y), x[3] = bf16hi_to_f32(v.y);
  x[4] = bf16lo_to_f32(v.z), x[5] = bf16hi_to_f32(v.z);
  x[6] = bf16lo_to_f32(v.w), x[7] = bf16hi_to_f32(v.w);
}

// D += A (16 tokens x 16 k, row) * B (16 k x 8 features, col); fragment layout of PTX mma.m16n8k16
__device__ __forceinline__ void mma16816(float* d, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// EPI as in gemm_tc.cu; LNIN: A is an un-normalised stream (QKV of layers >= 1, FFN-up); NBLK: 32-element K blocks per warp.
// blockIdx.y = which 32 tokens: a second pass runs on other SMs instead of after the first (one after the other, each pass
// cost its own chain of load -> MMA -> shared-memory sum -> residual load -> store, ~2.8 us per launch: r02ai)
template <int EPI, bool LNIN, int NBLK, int kH>
__global__ void __launch_bounds__(32 * max_warps(kH, NBLK), 1)
skinny_linear_kernel(const SkinnyParams p) {
  constexpr int kMaxWarps = max_warps(kH, NBLK);
  __shared__ float s_rs[32], s_nmr[32];                    // LayerNorm of a row of this CTA's 32: y = x * rs + nmr
  const int m0 = (int)blockIdx.y * 32;
  __shared__ float s_part[kMaxWarps][2][4][32];            // K-split partial sums [warp][tile][fragment register][lane]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const int r = lane >> 2, q = lane & 3;                   // fragment coordinates: row group, thread in group
  const int kq = warp % p.ks, group = warp / p.ks;
  const int n0 = ((int)blockIdx.x * p.fw + group) * 8;
  const int k0 = kq * NBLK * 32 + q * 8;                   // this lane's 8 elements of K block 0
  constexpr bool with_res = EPI == EPI_BIAS_RESIDUAL;

  // the warp's 8 x (32 NBLK) slice of W: constants, fetched while the previous kernel may still be running
  uint4 w[NBLK];
  {
    const __nv_bfloat16* wrow = p.W + (size_t)(n0 + r) * p.K + k0;
#pragma unroll
    for (int b = 0; b < NBLK; ++b) w[b] = __ldg(reinterpret_cast<const uint4*>(wrow + b * 32));
  }
  float bias[2], v2[2] = {1.0f, 1.0f};
#pragma unroll
  for (int f = 0; f < 2; ++f) {
    bias[f] = __ldg(p.bias + n0 + 2 * q + f);
    if (p.vec2) v2[f] = __ldg(p.vec2 + n0 + 2 * q + f);
  }
  ptx::griddep_launch();
  ptx::griddep_wait();

  // row statistics of the stream that goes through a LayerNorm here: A (LNIN) or the residual (vec2 given)
  const bool res_ln = with_res && p.vec2 != nullptr;
  if (LNIN || res_ln) {
    // eight lanes per row, four rows per warp at a time, a lane's twelve 16-byte loads all in flight together: one L2
    // round trip per 4 x nwarps rows (a warp per row, one row after the other, cost 2 - 4 us per launch at 12 tokens
    // and 16 us at 64: r02aa)
    const __nv_bfloat16* src = LNIN ? p.A : p.res;   // both have rows of kH elements in that case
    const int sub = lane & 7, slot = lane >> 3;
    const int m_end = min(p.M, m0 + 32);
    for (int mb = m0; mb < m_end; mb += 4 * nwarps) {
      const int m = mb + 4 * warp + slot;
      const __nv_bfloat16* row = src + (size_t)min(m, p.M - 1) * kH + sub * 8;
      uint4 v[kH / 64];
#pragma unroll
      for (int j = 0; j < kH / 64; ++j) v[j] = *reinterpret_cast<const uint4*>(row + j * 64);
      float s = 0.f, ss = 0.f;
#pragma unroll
      for (int j = 0; j < kH / 64; ++j) {
        float x[8];
        unpack8(v[j], x);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          s += x[e];
          ss = fmaf(x[e], x[e], ss);
        }
      }
#pragma unroll
      for (int off = 4; off > 0; off >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, off);
        ss += __shfl_xor_sync(0xffffffffu, ss, off);
      }
      if (sub == 0 && m < m_end) {
        const float mu = s * (1.0f / kH);
        const float rs = rsqrtf(fmaxf(fmaf(-mu, mu, ss * (1.0f / kH)), 0.0f) + p.eps);
        s_rs[m - m0] = rs;
        s_nmr[m - m0] = -mu * rs;
      }
    }
  }
  __syncthreads();

  {
    // two tiles of 16 tokens; rows past M re-read row M - 1 (their results are never stored)
    // two accumulator sets per tile (the two MMAs of a K block): half the length of the dependent MMA chain
    float acc[2][4], acc2[2][4];
#pragma unroll
    for (int t = 0; t < 2; ++t)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[t][i] = acc2[t][i] = 0.f;
    const bool two = m0 + 16 < p.M;   // warp-uniform
    const __nv_bfloat16* a0 = p.A + (size_t)min(m0 + r, p.M - 1) * p.K + k0;
    const __nv_bfloat16* a1 = p.A + (size_t)min(m0 + r + 8, p.M - 1) * p.K + k0;
    if (!two) {
#pragma unroll
      for (int b = 0; b < NBLK; ++b) {
        const uint4 ua = *reinterpret_cast<const uint4*>(a0 + b * 32);
        const uint4 ub = *reinterpret_cast<const uint4*>(a1 + b * 32);
        mma16816(acc[0], ua.x, ub.x, ua.y, ub.y, w[b].x, w[b].y);
        mma16816(acc2[0], ua.z, ub.z, ua.w, ub.w, w[b].z, w[b].w);
      }
    } else {
      const __nv_bfloat16* a2 = p.A + (size_t)min(m0 + 16 + r, p.M - 1) * p.K + k0;
      const __nv_bfloat16* a3 = p.A + (size_t)min(m0 + 24 + r, p.M - 1) * p.K + k0;
#pragma unroll
      for (int b = 0; b < NBLK; ++b) {
        const uint4 ua = *reinterpret_cast<const uint4*>(a0 + b * 32);
        const uint4 ub = *reinterpret_cast<const uint4*>(a1 + b * 32);
        const uint4 uc = *reinterpret_cast<const uint4*>(a2 + b * 32);
        const uint4 ud = *reinterpret_cast<const uint4*>(a3 + b * 32);
        mma16816(acc[0], ua.x, ub.x, ua.y, ub.y, w[b].x, w[b].y);
        mma16816(acc2[0], ua.z, ub.z, ua.w, ub.w, w[b].z, w[b].w);
        mma16816(acc[1], uc.x, ud.x, uc.y, ud.y, w[b].x, w[b].y);
        mma16816(acc2[1], uc.z, ud.z, uc.w, ud.w, w[b].z, w[b].w);
      }
    }
#pragma unroll
    for (int t = 0; t < 2; ++t)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[t][i] += acc2[t][i];
    if (p.ks > 1) {
#pragma unroll
      for (int t = 0; t < 2; ++t)
#pragma unroll
        for (int i = 0; i < 4; ++i) s_part[warp][t][i][lane] = acc[t][i];
      __syncthreads();
      if (kq == 0) {
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float y = 0.f;
            for (int s = 0; s < p.ks; ++s) y += s_part[warp + s][t][i][lane];   // fixed order: deterministic
            acc[t][i] = y;
          }
      }
    }
    if (kq == 0) {
      // fragment register i of tile t: token m0 + 16 t + r + 8 (i / 2), feature n0 + 2 q + (i % 2)
#pragma unroll
      for (int t = 0; t < 2; ++t)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int m = m0 + 16 * t + r + 8 * h;
          if (m < p.M) {
            float rs = 1.0f, nmr = 0.0f;
            if (LNIN || res_ln) rs = s_rs[m - m0], nmr = s_nmr[m - m0];
            float o[2];
#pragma unroll
            for (int f = 0; f < 2; ++f) {
              const float y = acc[t][2 * h + f];
              float x = LNIN ? fmaf(y, rs, fmaf(nmr, v2[f], bias[f])) : y + bias[f];
              if (EPI == EPI_BIAS_GELU) x = gelu_erf(x);
              if (with_res) {
                const float rv = __bfloat162float(p.res[(size_t)m * p.N + n0 + 2 * q + f]);
                x = fmaf(fmaf(rv, rs, nmr), v2[f], x);   // plain residual: rs = 1, nmr = 0, v2 = 1
              }
              o[f] = x;
            }
            *reinterpret_cast<__nv_bfloat162*>(p.out + (size_t)m * p.N + n0 + 2 * q) = __floats2bfloat162_rn(o[0], o[1]);
          }
        }
    }
  }
}

template <int EPI, bool LNIN, int NBLK, int kH>
int launch_variant(const SkinnyParams& p, cudaStream_t st) {
  ICD_CUDA(launch_chained(skinny_linear_kernel<EPI, LNIN, NBLK, kH>, dim3(p.N / (8 * p.fw), (p.M + 31) / 32), dim3(32 * p.ks * p.fw), 0, st,
                          1, p));
  count_launch();
  return ICD_OK;
}

}  // namespace

// 0 = never, 1 = forwards of at most kAutoTokens tokens, 2 = everything the kernel supports (the same 64 today; tests)
constexpr int kAutoTokens = 64;
static int g_encoder_skinny = 1;
int encoder_skinny() { return g_encoder_skinny; }
void encoder_set_skinny(int mode) { g_encoder_skinny = mode < 0 ? 0 : (mode > 2 ? 2 : mode); }
int skinny_max_tokens() { return g_encoder_skinny == 2 ? kMaxTokens : (g_encoder_skinny == 1 ? kAutoTokens : 0); }

// CTA shape of a launch: K blocks per warp, K splits and feature groups per CTA.  More than 16 tokens: K / 256 warps per
// feature group of 8 (short K ranges keep a tile's activation loads all in flight); wide outputs (QKV, FFN-up) take four
// groups per CTA (12 warps, 72 / 96 CTAs per 32 tokens at 768), H outputs one (O: 3 warps, FFN-down: 12; 96 CTAs).  Up to
// 16 tokens (one tile): one warp per group over one_tile_blocks(H) * 32 elements of K (4 warps per CTA at 768, FFN-down 4 K
// ranges) -- fewer partial sums to meet in shared memory; measured 0.337 vs 0.364 ms per 12-token forward (r02ac / r02ai),
// and the other way round from 24 tokens on (0.49 vs 0.43).  The O projection (N = K = H) keeps K ranges of 256.
static bool skinny_shape(int M, int N, int K, int H, int* nblk, int* ks, int* fw) {
  if ((H != 768 && H != 1024) || M < 1 || M > kMaxTokens || N % 32 != 0) return false;
  if (K != 768 && K != 1024 && K != 3072 && K != 4096) return false;
  int nb = (M <= 16 && !(N == H && K == H)) ? one_tile_blocks(H) : kBlk;
  if (K % (32 * nb) != 0) nb = kBlk;
  *nblk = nb;
  *ks = K / (32 * nb);
  *fw = N > H ? 4 : 1;
  return *ks * *fw <= max_warps(H, nb);
}

bool skinny_linear_supported(int M, int N, int K, int hidden) {
  int nblk, ks, fw;
  return skinny_shape(M, N, K, hidden, &nblk, &ks, &fw);
}

template <int kH, int kOne>
static int launch_width(const SkinnyParams& p, int epi, bool lnin, int nblk, cudaStream_t st) {
  switch (epi) {
    case EPI_BIAS:
      if (nblk == kOne)
        return lnin ? launch_variant<EPI_BIAS, true, kOne, kH>(p, st) : launch_variant<EPI_BIAS, false, kOne, kH>(p, st);
      return lnin ? launch_variant<EPI_BIAS, true, kBlk, kH>(p, st) : launch_variant<EPI_BIAS, false, kBlk, kH>(p, st);
    case EPI_BIAS_GELU:
      if (!lnin) break;
      return nblk == kOne ? launch_variant<EPI_BIAS_GELU, true, kOne, kH>(p, st) : launch_variant<EPI_BIAS_GELU, true, kBlk, kH>(p, st);
    case EPI_BIAS_RESIDUAL:
      if (lnin) break;
      return nblk == kOne ? launch_variant<EPI_BIAS_RESIDUAL, false, kOne, kH>(p, st)
                          : launch_variant<EPI_BIAS_RESIDUAL, false, kBlk, kH>(p, st);
  }
  set_error("skinny_linear: no kernel for epilogue %d (lnin %d) at N=%d K=%d", epi, lnin ? 1 : 0, p.N, p.K);
  return ICD_E_UNSUPPORTED;
}

int launch_skinny_linear(const SkinnyArgs& a, cudaStream_t st) {
  int nblk = 0, ks = 0, fw = 0;
  if (!skinny_shape(a.M, a.N, a.K, a.hidden, &nblk, &ks, &fw)) {
    set_error("skinny_linear: unsupported shape M=%d N=%d K=%d hidden=%d", a.M, a.N, a.K, a.hidden);
    return ICD_E_ARG;
  }
  const bool lnin = a.lnin != 0;
  if ((lnin && (a.K != a.hidden || !a.vec2)) || (a.epi == EPI_BIAS_RESIDUAL && (!a.res || (a.vec2 && a.N != a.hidden)))) {
    set_error("skinny_linear: LayerNorm statistics cover rows of %d elements", a.hidden);
    return ICD_E_ARG;
  }
  SkinnyParams p{};
  p.A = reinterpret_cast<const __nv_bfloat16*>(a.A);
  p.W = reinterpret_cast<const __nv_bfloat16*>(a.W);
  p.bias = a.bias;
  p.vec2 = a.vec2;
  p.res = reinterpret_cast<const __nv_bfloat16*>(a.res);
  p.out = reinterpret_cast<__nv_bfloat16*>(a.out);
  p.M = a.M, p.N = a.N, p.K = a.K;
  p.eps = a.eps;
  p.ks = ks;
  p.fw = fw;
  return a.hidden == 768 ? launch_width<768, one_tile_blocks(768)>(p, a.epi, lnin, nblk, st)
                         : launch_width<1024, one_tile_blocks(1024)>(p, a.epi, lnin, nblk, st);
}

}  // namespace icd
