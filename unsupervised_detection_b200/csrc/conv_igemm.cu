// tcgen05 implicit-GEMM convolution engine for sm_100a (forward / data-gradient / transposed conv / weight-gradient).
//
// Replaces the TF1 op classes K1/K3/K5/K6 of SURVEY.md section 2.2 (tf.layers.conv2d, tf.nn.conv2d,
// tf.layers.conv2d_transpose and their tf.gradients twins; reference call sites
// models/utils/convolution_utils.py:46,81 and models/PWCNet/model_pwcnet.py:161-165,286,484-504,562-574).
//
// Design (see DESIGN.md): one CTA = one 128-row tile of the GEMM (rows = output pixels).  Four producer warps gather the
// im2col A tile (128 rows x 64 bf16 of K) and the packed-weight B tile straight into the canonical SWIZZLE_128B K-major
// shared-memory layout with 16-byte cp.async (zero-fill = SAME padding); one thread of a fifth warp issues
// tcgen05.mma.kind::f16 (M=128, N=BN, K=16) with the fp32 accumulator in TMEM; smem stages are recycled with
// tcgen05.commit -> mbarrier.  The producer warps then become the epilogue: tcgen05.ld the accumulator, apply
// bias / residuals / activation and store bf16 and/or fp32 NHWC.
#include "ptx.cuh"
#include "../../include/cis_b200.h"
#include "common.cuh"
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

// cp.async (LDGSTS) writes shared memory through the generic proxy while tcgen05.mma reads it through the async proxy.  Every
// cp.async producer therefore publishes a stage itself: commit_group, wait_group<lag> (its own copies of the stage landed),
// fence.proxy.async, then a plain mbarrier.arrive -- the MMA warp needs no fence.  The lag keeps (stages - 1) groups in flight.

namespace cis {

// Developer-only pipeline trace (make trace -> libcis_b200_trace.so, tools/trace_conv.py): CTA (0,0,0) records SM-clock stamps of its
// MMA-issue loop so per-step wait / issue time can be read back.  Compiled out of the product library.
#ifdef CIS_TRACE
__device__ unsigned long long* g_trace = nullptr;
__device__ int g_trace_cap = 0;
#define CIS_TRACE_AT(slot)                                                                                         \
  do {                                                                                                             \
    if (g_trace && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && (slot) < g_trace_cap) g_trace[(slot)] = clock64(); \
  } while (0)
#else
#define CIS_TRACE_AT(slot) ((void)0)
#endif

static constexpr int kBM = 128;       // GEMM rows per CTA
static constexpr int kBK = 64;        // bf16 K elements per stage (128-byte swizzled rows)
static constexpr int kAStage = kBM * 128;
static constexpr int kThreads = 160;  // halo / wgrad kernels: 4 producer/epilogue warps + 1 MMA warp
// conv_halo_kernel<BN>: warps 0-3 producers + epilogue; BN >= 64 adds warps 4-7 (epilogue only: the wide epilogue is instruction-bound on its
// warps); last warp = MMA issuer / TMEM owner.  BN <= 32 keeps 160 threads: there the number of co-resident CTAs matters more (measured).
template <int BN> struct HaloCfg {
  static constexpr int kMmaWarp = BN >= 64 ? 8 : 4;
  static constexpr int kThreads = (kMmaWarp + 1) * 32;
  static constexpr int kMinCtas = BN >= 64 ? 2 : (BN == 32 ? 3 : 4);
};
static constexpr int kGProducers = 256;   // gather kernel: 8 producer/epilogue warps (its cp.async address arithmetic is the bottleneck)
static constexpr int kGThreads = 288;     // + 1 MMA warp

struct SrcS {
  const __nv_bfloat16* ptr;
  int pitch, c_off, chunks, n_mod;
};


// One 16-column chunk of the fused epilogue: bias -> (+bf16 accumulate | +fp32 residual) -> activation -> (+skip) -> stores.
__device__ __forceinline__ void epi_chunk(const CisConv& p, float (&v)[16], const int cg, const size_t dpix) {
  if (p.bias) {
#pragma unroll
    for (int e = 0; e < 16; ++e) v[e] += __ldg(p.bias + cg + e);
  }
  if (p.add_pre && cg < p.out_ch) {
    const uint4* a = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.add_pre) + dpix * p.add_pre_pitch +
                                                    p.add_pre_coff + cg);
    const int nv = (p.out_ch - cg >= 16) ? 2 : 1;
    for (int h2 = 0; h2 < nv; ++h2) {
      const uint4 u = __ldg(a + h2);
      const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        v[h2 * 8 + 2 * e] += bf16lo(w4[e]);
        v[h2 * 8 + 2 * e + 1] += bf16hi(w4[e]);
      }
    }
  }
  if (p.addf_pre) {
    for (int e = 0; e < 16 && cg + e < p.outf_ch; ++e) v[e] += __ldg(p.addf_pre + dpix * p.addf_pitch + p.addf_coff + cg + e);
  }
  if (p.act == CIS_ACT_ELU) {
#pragma unroll
    for (int e = 0; e < 16; ++e) v[e] = v[e] > 0.f ? v[e] : expm1f(v[e]);
  } else if (p.act == CIS_ACT_LEAKY) {
#pragma unroll
    for (int e = 0; e < 16; ++e) v[e] = v[e] > 0.f ? v[e] : v[e] * p.alpha;
  }
  if (p.add_post && cg < p.out_ch) {
    const uint4* a = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.add_post) + dpix * p.add_post_pitch +
                                                    p.add_post_coff + cg);
    const int nv = (p.out_ch - cg >= 16) ? 2 : 1;
    for (int h2 = 0; h2 < nv; ++h2) {
      const uint4 u = __ldg(a + h2);
      const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        v[h2 * 8 + 2 * e] += bf16lo(w4[e]);
        v[h2 * 8 + 2 * e + 1] += bf16hi(w4[e]);
      }
    }
  }
  if (p.mode == 1) {
    if (cg == 0) p.outf[dpix] = 1.f / (1.f + __expf(-(v[0] - v[1]) * 0.1f));
    return;
  }
  if (p.out && cg < p.out_ch) {
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) + dpix * p.out_pitch + p.out_coff + cg;
    if (((p.out_ch | p.out_coff | p.out_pitch) & 7) == 0) {
      uint4 u0 = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
      *reinterpret_cast<uint4*>(o) = u0;
      if (p.out_ch - cg >= 16) {
        uint4 u1 = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
        *reinterpret_cast<uint4*>(o + 8) = u1;
      }
    } else {
      for (int e = 0; e < 16 && cg + e < p.out_ch; ++e) o[e] = __float2bfloat16(v[e]);
    }
  }
  if (p.outf && cg < p.outf_ch) {
    float* o = p.outf + dpix * p.outf_pitch + p.outf_coff + cg;
    for (int e = 0; e < 16 && cg + e < p.outf_ch; ++e) o[e] = v[e];
  }
}



// Latency-batched epilogue for NC x 16 accumulator columns of one row: residual loads are issued first, then all TMEM loads,
// ONE wait, then the arithmetic and the stores (the per-chunk version paid a full TMEM + global-load round trip per 16 columns).
template <int NC>
__device__ __forceinline__ void epi_group(const CisConv& p, const uint32_t taddr, const int cg0, const size_t dpix, const bool valid,
                                          const float* __restrict__ sbias) {
  // one residual operand per launch: add_pre (gradient accumulation, before the activation) or add_post (skip, after it)
  uint4 rres[NC][2];
  const bool is_pre = p.add_pre != nullptr;
  const __nv_bfloat16* rp = reinterpret_cast<const __nv_bfloat16*>(is_pre ? p.add_pre : p.add_post);
  const bool has_res = valid && rp != nullptr;
  const size_t roff = has_res ? (dpix * (is_pre ? p.add_pre_pitch : p.add_post_pitch) + (is_pre ? p.add_pre_coff : p.add_post_coff)) : 0;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int cg = cg0 + 16 * c;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      rres[c][h] = make_uint4(0, 0, 0, 0);
      if (has_res && cg + 8 * h < p.out_ch) rres[c][h] = __ldg(reinterpret_cast<const uint4*>(rp + roff + cg) + h);
    }
  }
  uint32_t raw[NC][16];
#pragma unroll
  for (int c = 0; c < NC; ++c) tmem_ld16_nowait(taddr + 16 * c, raw[c]);
  tmem_ld_wait();
  if (!valid) return;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int cg = cg0 + 16 * c;
    float v[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) v[e] = __uint_as_float(raw[c][e]);
    if (p.bias) {
      const float4* sb = reinterpret_cast<const float4*>(sbias + (cg - cg0));   // sbias = this group's first column; 16-float aligned: 4 x LDS.128
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 b4 = sb[q];
        v[4 * q] += b4.x; v[4 * q + 1] += b4.y; v[4 * q + 2] += b4.z; v[4 * q + 3] += b4.w;
      }
    }
    if (is_pre) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint32_t w4[4] = {rres[c][h].x, rres[c][h].y, rres[c][h].z, rres[c][h].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          v[h * 8 + 2 * e] += bf16lo(w4[e]);
          v[h * 8 + 2 * e + 1] += bf16hi(w4[e]);
        }
      }
    }
    if (p.addf_pre) {
      for (int e = 0; e < 16 && cg + e < p.outf_ch; ++e) v[e] += __ldg(p.addf_pre + dpix * p.addf_pitch + p.addf_coff + cg + e);
    }
    if (p.act == CIS_ACT_ELU) {
      // exp through MUFU.EX2 (4 instructions per element instead of the ~40 of expm1f): |error| <= ~1e-7 absolute, far below the
      // bf16 rounding of the stored activation; the epilogue runs on one warp per scheduler, so instruction count IS its time
#pragma unroll
      for (int e = 0; e < 16; ++e) v[e] = v[e] > 0.f ? v[e] : __expf(v[e]) - 1.f;
    } else if (p.act == CIS_ACT_LEAKY) {
#pragma unroll
      for (int e = 0; e < 16; ++e) v[e] = v[e] > 0.f ? v[e] : v[e] * p.alpha;
    }
    if (!is_pre) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint32_t w4[4] = {rres[c][h].x, rres[c][h].y, rres[c][h].z, rres[c][h].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          v[h * 8 + 2 * e] += bf16lo(w4[e]);
          v[h * 8 + 2 * e + 1] += bf16hi(w4[e]);
        }
      }
    }
    if (p.mode == 1) {
      if (cg == 0) p.outf[dpix] = 1.f / (1.f + __expf(-(v[0] - v[1]) * 0.1f));
      continue;
    }
    if (p.out && cg < p.out_ch) {
      __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) + dpix * p.out_pitch + p.out_coff + cg;
      if (((p.out_ch | p.out_coff | p.out_pitch) & 7) == 0) {
        *reinterpret_cast<uint4*>(o) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
        if (p.out_ch - cg >= 16)
          *reinterpret_cast<uint4*>(o + 8) =
              make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
      } else {
        for (int e = 0; e < 16 && cg + e < p.out_ch; ++e) o[e] = __float2bfloat16(v[e]);
      }
    }
    if (p.outf && cg < p.outf_ch) {
      float* o = p.outf + dpix * p.outf_pitch + p.outf_coff + cg;
      for (int e = 0; e < 16 && cg + e < p.outf_ch; ++e) o[e] = v[e];
    }
  }
}
// columns [c_lo, c_hi) of one row (multiples of 16), in groups of 32 columns (register budget); sbias: the BN columns of THIS n-tile
template <int BN>
__device__ __forceinline__ void epi_cols(const CisConv& p, const uint32_t t_row, const int cbase, const size_t dpix, const bool valid,
                                         const float* __restrict__ sbias, const int c_lo, const int c_hi) {
  int c0 = c_lo;
#pragma unroll 1
  for (; c0 + 32 <= c_hi; c0 += 32) epi_group<2>(p, t_row + c0, cbase + c0, dpix, valid, sbias + c0);
  if (c0 < c_hi) epi_group<1>(p, t_row + c0, cbase + c0, dpix, valid, sbias + c0);
}
// all BN columns of one row
template <int BN>
__device__ __forceinline__ void epi_row(const CisConv& p, const uint32_t t_row, const int cbase, const size_t dpix, const bool valid,
                                        const float* __restrict__ sbias) {
  epi_cols<BN>(p, t_row, cbase, dpix, valid, sbias, 0, BN);
}

// ---- split-K (two launches): every CTA of a tile stores its partial accumulator to a private fp32 slice; splitk_finish_kernel sums the
// slices in a fixed order and runs the fused epilogue.
template <int BN>
__device__ __forceinline__ void splitk_store_partial(float* slice, uint32_t t_row, int row, int c_lo = 0, int c_hi = BN) {
  // slice = this split's private fp32 tile, stored as float4 COLUMNS: element (row, c) at ((c / 4) * 128 + row) * 4 + c % 4.  A warp
  // (32 consecutive accumulator rows, same columns) then writes 512 contiguous bytes per store instruction; the row-major layout of
  // r01/r02 made every st.v4 touch 32 different 128-byte lines and the LSU, not HBM, bounded the epilogue (~10k clk per 128x128 tile
  // in the CIS_TRACE build -- as long as the whole MMA loop of a split).  No atomics, fixed summation order later.
#pragma unroll 1
  for (int c0 = c_lo; c0 < c_hi; c0 += 16) {
    float v[16];
    tmem_ld16(t_row + c0, v);
    float4* o = reinterpret_cast<float4*>(slice) + (size_t)(c0 / 4) * kBM + row;
    o[0] = make_float4(v[0], v[1], v[2], v[3]);
    o[kBM] = make_float4(v[4], v[5], v[6], v[7]);
    o[2 * kBM] = make_float4(v[8], v[9], v[10], v[11]);
    o[3 * kBM] = make_float4(v[12], v[13], v[14], v[15]);
  }
}
// sum of the nsplit private slices of one tile for (row, c0..c0+15); loads are plain L2 loads (__ldcg) issued in batches of
// 4 slices x 4 float4 so their latencies overlap (a volatile-asm version serialised ~150 round trips per thread: ncu r01d)
template <int BN>
__device__ __forceinline__ void splitk_reduce16(const float* tile0, int nsplit, int row, int c0, float* v) {
#pragma unroll
  for (int e = 0; e < 16; ++e) v[e] = 0.f;
  const float4* q0 = reinterpret_cast<const float4*>(tile0) + (size_t)(c0 / 4) * kBM + row;    // float4-column layout of splitk_store_partial
  const size_t zstride = (size_t)kBM * BN / 4;
  int z = 0;
  for (; z + 4 <= nsplit; z += 4) {
    float4 t[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int h = 0; h < 4; ++h) t[u][h] = __ldcg(q0 + (size_t)(z + u) * zstride + h * kBM);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        v[4 * h] += t[u][h].x; v[4 * h + 1] += t[u][h].y; v[4 * h + 2] += t[u][h].z; v[4 * h + 3] += t[u][h].w;
      }
  }
  for (; z < nsplit; ++z) {
    float4 t[4];
#pragma unroll
    for (int h = 0; h < 4; ++h) t[h] = __ldcg(q0 + (size_t)z * zstride + h * kBM);
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      v[4 * h] += t[h].x; v[4 * h + 1] += t[h].y; v[4 * h + 2] += t[h].z; v[4 * h + 3] += t[h].w;
    }
  }
}
// Cluster split-K: every CTA of the cluster has written its partial tile to its own shared memory as float4 columns
// stage[(c4 * 128 + row)] (conflict-free: lanes = consecutive rows).  CTA `rank` of `S` then owns accumulator rows
// [rank * rpc, (rank + 1) * rpc): it sums the S partials in rank order (deterministic) through DSMEM and runs the fused epilogue.
template <int BN, typename DPIX>
__device__ __forceinline__ void cluster_reduce_rows(const CisConv& p, const uint32_t stage, const int S, const int rank, const int tid,
                                                    const int nthreads, const int cbase, DPIX dpix_of) {
  const int rpc = (kBM + S - 1) / S;
  const int r0 = rank * rpc, r1 = min(kBM, r0 + rpc);
  constexpr int G16 = BN / 16;
  for (int it = tid; it < (r1 - r0) * G16; it += nthreads) {
    const int row = r0 + it / G16, c0 = (it % G16) * 16;
    float v[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) v[e] = 0.f;
    for (int q = 0; q < S; ++q) {
      const uint32_t base = dsmem_addr(stage, (uint32_t)q);
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const float4 t = dsmem_ld4(base + (uint32_t)(((c0 / 4 + h) * kBM + row) * 16));
        v[4 * h] += t.x; v[4 * h + 1] += t.y; v[4 * h + 2] += t.z; v[4 * h + 3] += t.w;
      }
    }
    bool valid;
    const size_t dpix = dpix_of(row, valid);
    if (valid) epi_chunk(p, v, cbase + c0, dpix);
  }
}
// this warp's 32 accumulator rows x columns [c_lo, c_hi) -> shared-memory stage in the layout above
__device__ __forceinline__ void tmem_to_stage(const uint32_t t_row, const int row, const uint32_t stage, const int c_lo, const int c_hi) {
#pragma unroll 1
  for (int c0 = c_lo; c0 < c_hi; c0 += 16) {
    float v[16];
    tmem_ld16(t_row + c0, v);
#pragma unroll
    for (int h = 0; h < 4; ++h)
      asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(stage + (uint32_t)(((c0 / 4 + h) * kBM + row) * 16)), "f"(v[4 * h]),
                   "f"(v[4 * h + 1]), "f"(v[4 * h + 2]), "f"(v[4 * h + 3])
                   : "memory");
  }
}

template <int BN>
struct FwdCfg {
  // kLag + 1 K blocks of gathers are in flight per producer thread (the im2col loads are L2 round trips of ~1 us).  A deeper ring
  // (5-6 stages for BN <= 32) was measured SLOWER: it drops the thin layers from 3 to 2 co-resident CTAs per SM.
  static constexpr int kStages = (BN == 128) ? 3 : 4;
  static constexpr int kLag = kStages - 2;
  static constexpr int kBStage = BN * 128;
  static constexpr int kSmem = kStages * (kAStage + kBStage) + 1024;
  static constexpr int kTmemCols = BN < 32 ? 32 : BN;
};

template <int BN>
__global__ void __launch_bounds__(kGThreads) conv_igemm_kernel(const __grid_constant__ CisConv p) {
  using Cfg = FwdCfg<BN>;
  constexpr int S = Cfg::kStages;
  constexpr int kMmaWarp = kGProducers / 32;
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bars[2 * S + 1];
  __shared__ uint32_t tmem_slot;
  __shared__ int s_dh[CIS_MAX_TAPS], s_dw[CIS_MAX_TAPS];
  __shared__ SrcS s_src[CIS_MAX_SRC];

  const uint32_t tile_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t a_base = tile_base;
  const uint32_t b_base = tile_base + S * kAStage;
  const uint32_t bar_full = smem_u32(&bars[0]);
  const uint32_t bar_empty = smem_u32(&bars[S]);
  const uint32_t bar_accum = smem_u32(&bars[2 * S]);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int M = p.N * p.OH * p.OW;
  const int m_chunks = [&] {
    int s = 0;
    for (int i = 0; i < p.nsrc; ++i) s += p.src[i].chunks;
    return s;
  }();
  const int nkb_all = p.K_pad / kBK;
  const int nsplit = p.splits > 1 ? p.splits : 1;
  const int kper = (nkb_all + nsplit - 1) / nsplit;
  const int kb_lo = blockIdx.z * kper;
  const int nkb = min(kper, nkb_all - kb_lo);     // host guarantees nkb >= 1 for every split
  const int ny = blockIdx.y;
  __shared__ __align__(16) float s_bias[BN];
  pdl_launch_dependents();

  if (tid < p.ntaps) {
    s_dh[tid] = p.dh[tid];
    s_dw[tid] = p.dw[tid];
  }
  if (tid < p.nsrc) {
    s_src[tid].ptr = reinterpret_cast<const __nv_bfloat16*>(p.src[tid].ptr);
    s_src[tid].pitch = p.src[tid].pitch;
    s_src[tid].c_off = p.src[tid].c_off;
    s_src[tid].chunks = p.src[tid].chunks;
    s_src[tid].n_mod = p.src[tid].n_mod;
  }
  if (warp == kMmaWarp) {
    if (lane == 0) {
      for (int s = 0; s < S; ++s) {
        mbar_init(bar_full + 8 * s, kGProducers);
        mbar_init(bar_empty + 8 * s, 1);
      }
      mbar_init(bar_accum, 1);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc<Cfg::kTmemCols>(smem_u32(&tmem_slot));
  }
  pdl_wait();   // everything above touched only kernel parameters / shared memory / TMEM
  if (tid < BN) s_bias[tid] = p.bias ? p.bias[ny * BN + tid] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  if (tid == 0) CIS_TRACE_AT(0);

  if (warp < kMmaWarp) {
    // ------------------------------------------------------------------ producers: thread = (16-byte K chunk j, rows rl + 32 i)
    const int j = tid & 7;          // 16-byte chunk within the 128-byte K row
    const int rl = tid >> 3;        // 0..31
    const uint32_t sw_off = (uint32_t)((j ^ (rl & 7)) << 4);
    // Per-row constants (this thread's 4 rows): top-left input pixel, and the linear pixel index of it in the plain and in the
    // batch-broadcast (n % n_mod) view of the sources.  The K loop below is division-free: r02's ncu source view showed the producer
    // warps issue-bound on the integer divisions / 64-bit address arithmetic of every (K block, row), not on the loads.
    int hb[4], wb[4], pre[4], prem[4];
    int nm0 = 0;                          // the batch-broadcast modulus (sources with n_mod > 0 share one; others: slow path)
    for (int i = 0; i < p.nsrc; ++i)
      if (p.src[i].n_mod > 0 && nm0 == 0) nm0 = p.src[i].n_mod;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int g = blockIdx.x * kBM + rl + 32 * i;
      if (g < M) {
        const int ow = g % p.OW;
        const int t = g / p.OW;
        const int oh = t % p.OH;
        const int n = t / p.OH;
        hb[i] = oh * p.sh;
        wb[i] = ow * p.sw;
        pre[i] = (n * p.H + hb[i]) * p.W + wb[i];
        prem[i] = ((nm0 ? n % nm0 : n) * p.H + hb[i]) * p.W + wb[i];
      } else {
        hb[i] = -(1 << 20);
        wb[i] = 0;
        pre[i] = prem[i] = 0;
      }
    }
    const __nv_bfloat16* wrow = reinterpret_cast<const __nv_bfloat16*>(p.wpack) + (size_t)(ny * BN + rl) * p.K_pad + j * 8;
    // (tap, channel chunk) of this thread's K chunk, advanced by 8 chunks per K block without dividing
    const int adv_t = 8 / m_chunks, adv_c = 8 - adv_t * m_chunks;
    int t = (kb_lo * 8 + j) / m_chunks, c = (kb_lo * 8 + j) - t * m_chunks;

    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % S;
      const uint32_t ph = (uint32_t)((kb / S) & 1);
      mbar_wait(bar_empty + 8 * s, ph ^ 1u);
      // ---- A: this thread's K chunk -> (tap t, source si, channel chunk cs)
      const bool kvalid = t < p.ntaps;
      const int tt = kvalid ? t : 0;
      int si = 0, cs = c;
      while (si < p.nsrc - 1 && cs >= s_src[si].chunks) {
        cs -= s_src[si].chunks;
        ++si;
      }
      const __nv_bfloat16* sp = s_src[si].ptr;
      const int pitch = s_src[si].pitch;
      const int nmod = s_src[si].n_mod;
      const int dh = s_dh[tt], dw = s_dw[tt];
      const int toff = dh * p.W + dw;
      const __nv_bfloat16* spc = sp + s_src[si].c_off + cs * 8;
      const bool slow_mod = nmod != 0 && nmod != nm0;
      const uint32_t a_dst = a_base + s * kAStage + rl * 128 + sw_off;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int h = hb[i] + dh, w = wb[i] + dw;
        const bool ok = kvalid && (unsigned)h < (unsigned)p.H && (unsigned)w < (unsigned)p.W;
        int pix = (nmod ? prem[i] : pre[i]) + toff;
        if (slow_mod) {                    // a second, different modulus: recompute (never the case in this model)
          const int n = (pre[i] / (p.H * p.W)) % nmod;
          pix = (n * p.H + h) * p.W + w;
        }
        cp_async16(a_dst + i * 32 * 128, ok ? (const void*)(spc + (size_t)pix * pitch) : (const void*)sp, ok ? 16u : 0u);
      }
      t += adv_t;
      c += adv_c;
      if (c >= m_chunks) {
        c -= m_chunks;
        ++t;
      }
      // ---- B: packed weights, rows rl + 32 i
      const uint32_t b_dst = b_base + s * Cfg::kBStage + rl * 128 + sw_off;
      if constexpr (BN >= 32) {
#pragma unroll
        for (int i = 0; i < BN / 32; ++i) cp_async16(b_dst + i * 32 * 128, wrow + (size_t)i * 32 * p.K_pad + (kb_lo + kb) * kBK, 16u);
      } else {
        if (rl < BN) cp_async16(b_dst, wrow + (kb_lo + kb) * kBK, 16u);
      }
      cp_async_commit();
      if (kb >= Cfg::kLag) {         // publish block kb-kLag (its copies have landed) while the kLag younger blocks are in flight
        cp_async_wait<Cfg::kLag>();
        fence_proxy_async();
        mbar_arrive(bar_full + 8 * ((kb - Cfg::kLag) % S));
      }
    }
#pragma unroll
    for (int i = Cfg::kLag - 1; i >= 0; --i) {   // drain: block nkb-1-i has i younger groups behind it
      if (nkb - 1 - i < 0) continue;
      if (i == 3) cp_async_wait<3>();
      else if (i == 2) cp_async_wait<2>();
      else if (i == 1) cp_async_wait<1>();
      else cp_async_wait<0>();
      fence_proxy_async();
      mbar_arrive(bar_full + 8 * ((nkb - 1 - i) % S));
    }

    // ------------------------------------------------------------------ epilogue: warps w and w + 4 share a TMEM lane quarter and split the columns
    mbar_wait(bar_accum, 0);
    tc_fence_after();
    if (tid == 0) CIS_TRACE_AT(2);
    const int qtr = warp & 3, half = warp >> 2;
    const int row = qtr * 32 + lane;
    const int g = blockIdx.x * kBM + row;
    const bool valid = g < M;
    size_t dpix = 0;
    if (valid) {
      const int ow = g % p.OW;
      const int t = g / p.OW;
      const int oh = t % p.OH;
      const int n = t / p.OH;
      dpix = (size_t)(n * p.DH + oh * p.osh + p.oa) * p.DW + ow * p.osw + p.ob;
    }
    const uint32_t t_row = tmem + ((uint32_t)(qtr * 32) << 16);
    const int cbase = ny * BN;
    constexpr int kHalf = BN >= 32 ? BN / 2 : BN;                 // BN = 16: the first warp group does it all
    const int c_lo = half * kHalf, c_hi = (BN >= 32 || half == 0) ? c_lo + kHalf : c_lo;
    if (nsplit > 1 && p.sk_cluster) {
      // cluster split-K: partial tile -> own shared memory (the operand ring is dead: every MMA has completed); reduced below
      tmem_to_stage(t_row, row, tile_base, c_lo, c_hi);
    } else if (nsplit > 1) {
      // two-launch split-K: this split's private fp32 slice; splitk_finish_kernel reduces the slices and runs the fused epilogue
      const int tile_id = blockIdx.x * gridDim.y + ny;
      float* tile0 = p.sk_scratch + (size_t)tile_id * nsplit * kBM * BN;
      splitk_store_partial<BN>(tile0 + (size_t)blockIdx.z * kBM * BN, t_row, row, c_lo, c_hi);
    } else {
      epi_cols<BN>(p, t_row, cbase, dpix, valid, s_bias, c_lo, c_hi);
    }
  } else {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = make_idesc_bf16(kBM, BN, 0, 0);
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % S;
      const uint32_t ph = (uint32_t)((kb / S) & 1);
      mbar_wait(bar_full + 8 * s, ph);
      tc_fence_after();
      if (elect_one()) {
        CIS_TRACE_AT(8 + 2 * kb);
        const uint32_t alo = desc_lo(a_base + s * kAStage, 16), blo = desc_lo(b_base + s * Cfg::kBStage, 16);
        const uint32_t dhi = desc_hi(1024);
#pragma unroll
        for (int k = 0; k < kBK / 16; ++k) umma_bf16_lh(tmem, alo + 2 * k, dhi, blo + 2 * k, dhi, idesc, (uint32_t)((kb | k) != 0));
        umma_commit(bar_empty + 8 * s);
        if (kb == nkb - 1) umma_commit(bar_accum);
        CIS_TRACE_AT(9 + 2 * kb);
      }
      __syncwarp();
    }
  }
  if (nsplit > 1 && p.sk_cluster) {
    cluster_sync_all();                       // every CTA's partial tile is in its shared memory
    if (warp < kMmaWarp) {
      const int cbase = ny * BN;
      cluster_reduce_rows<BN>(p, tile_base, nsplit, (int)cluster_ctarank(), tid, kGProducers, cbase, [&](int row, bool& valid) -> size_t {
        const int g = blockIdx.x * kBM + row;
        valid = g < M;
        if (!valid) return 0;
        const int ow = g % p.OW;
        const int t = g / p.OW;
        const int oh = t % p.OH;
        const int n = t / p.OH;
        return (size_t)(n * p.DH + oh * p.osh + p.oa) * p.DW + ow * p.osw + p.ob;
      });
    }
    cluster_sync_all();                       // peers may still be reading this CTA's shared memory
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0) CIS_TRACE_AT(3);
  if (warp == kMmaWarp) tmem_dealloc<Cfg::kTmemCols>(tmem);
}


// ======================================================================================================= halo-resident conv
// Stride-1 gathers (forward convs incl. dilated ones, stride-1 data gradients, parity launches of stride-2 data gradients and
// of the 4x4 s2 transposed convs).  The CTA owns MT stacked tiles of 16x8 output pixels of one dilation phase; per 64-channel
// chunk the (16*MT+ey) x (8+ex) input halo is copied ONCE into shared memory (SWIZZLE_128B rows of 128 B = one pixel x 64 ch)
// and every tap (dy,dx) reads it in place: A descriptor start = halo + ((16*m+dy)*Wh + dx)*128, SBO = Wh*128.  The hardware
// applies the 128B swizzle on absolute shared-memory address bits (tools/umma_probe.cu), so 128-byte-granular starts and a
// non-1024 SBO are legal with base_offset = 0.  im2col traffic drops from k*k x to ~1.3 x and the packed weights of a
// (tap, chunk) are reused by the MT tiles.
static constexpr int kHaloMaxBStages = 8;
// compact thin halo: bytes between the 8-channel planes of one halo stage (16 B per pixel, 128-byte aligned planes)
__host__ __device__ __forceinline__ uint32_t thin_plane_bytes(int HP) { return ((uint32_t)HP * 16u + 127u) & ~127u; }
struct HaloMaps {
  // one 4-D (C, W, H, N) SWIZZLE_128B map per (concat source, stride-2 phase): index si * nph + phase; box = (64, Wh, Hh, 1)
  CUtensorMap m[CIS_MAX_SRC * 4];
};

// MMAs of one weight stage (gt taps of one 64-channel chunk, MT stacked tiles, NK K=16 steps each), issued by ONE thread.  The tap
// offsets come from a shared-memory table; the next tap's offset is fetched BEFORE the current tap's MMAs are issued so the
// LDS -> R2UR -> descriptor chain (~100 clk, measured 220 clk per single-MMA tap in r02) overlaps the previous issue.
// MT == 1 (every thin layer): straight-line groups of four taps -- the four tap offsets of the NEXT group are loaded before this group's
// MMAs are issued, no per-tap branch or tile loop.  (r02 trace: the generic loop below cost 105-157 clk per single-MMA tap, 3-4x the
// 36 clk the tensor pipe needs for a 128x16x16 MMA; the thin layers were bound by this thread, not by shared memory.)
template <int NK>
__device__ __forceinline__ void halo_issue_mt1(const uint32_t tmem, const uint32_t hlo, uint32_t blo, const uint32_t* s_aoff, const int gt,
                                               const uint32_t bstep, const uint32_t ahi, const uint32_t bhi, const uint32_t idesc,
                                               const bool first) {
  int tt = 0;
  uint32_t acc = first ? 0u : 1u;
  uint32_t o0 = 0, o1 = 0, o2 = 0, o3 = 0;
  if (gt >= 4) {
    o0 = s_aoff[0];
    o1 = s_aoff[1];
    o2 = s_aoff[2];
    o3 = s_aoff[3];
  }
  for (; tt + 4 <= gt; tt += 4) {
    const uint32_t a0 = hlo + o0, a1 = hlo + o1, a2 = hlo + o2, a3 = hlo + o3;
    if (tt + 8 <= gt) {
      o0 = s_aoff[tt + 4];
      o1 = s_aoff[tt + 5];
      o2 = s_aoff[tt + 6];
      o3 = s_aoff[tt + 7];
    }
#pragma unroll
    for (int k = 0; k < NK; ++k) umma_bf16_lh(tmem, a0 + 2 * k, ahi, blo + 2 * k, bhi, idesc, k ? 1u : acc);
#pragma unroll
    for (int k = 0; k < NK; ++k) umma_bf16_lh(tmem, a1 + 2 * k, ahi, blo + bstep + 2 * k, bhi, idesc, 1u);
#pragma unroll
    for (int k = 0; k < NK; ++k) umma_bf16_lh(tmem, a2 + 2 * k, ahi, blo + 2 * bstep + 2 * k, bhi, idesc, 1u);
#pragma unroll
    for (int k = 0; k < NK; ++k) umma_bf16_lh(tmem, a3 + 2 * k, ahi, blo + 3 * bstep + 2 * k, bhi, idesc, 1u);
    acc = 1u;
    blo += 4 * bstep;
  }
  if (tt < gt) {              // 1-3 left-over taps
    const uint32_t r0 = s_aoff[tt], r1 = tt + 1 < gt ? s_aoff[tt + 1] : 0u, r2 = tt + 2 < gt ? s_aoff[tt + 2] : 0u;
#pragma unroll
    for (int k = 0; k < NK; ++k) umma_bf16_lh(tmem, hlo + r0 + 2 * k, ahi, blo + 2 * k, bhi, idesc, k ? 1u : acc);
    if (tt + 1 < gt) {
#pragma unroll
      for (int k = 0; k < NK; ++k) umma_bf16_lh(tmem, hlo + r1 + 2 * k, ahi, blo + bstep + 2 * k, bhi, idesc, 1u);
    }
    if (tt + 2 < gt) {
#pragma unroll
      for (int k = 0; k < NK; ++k) umma_bf16_lh(tmem, hlo + r2 + 2 * k, ahi, blo + 2 * bstep + 2 * k, bhi, idesc, 1u);
    }
  }
}

template <int NK>
__device__ __forceinline__ void halo_issue_stage(const uint32_t tmem, const uint32_t hlo, uint32_t blo, const uint32_t* s_aoff, const int gt,
                                                 const int MT, const int BN, const uint32_t ahi, const uint32_t bhi, const uint32_t a_mstep,
                                                 const uint32_t bstep, const uint32_t idesc, const bool first) {
  if (NK == 1 && MT == 1) {      // single-MMA taps: the loop overhead below would dominate
    halo_issue_mt1<NK>(tmem, hlo, blo, s_aoff, gt, bstep, ahi, bhi, idesc, first);
    return;
  }
  uint32_t off0 = s_aoff[0], off1 = gt > 1 ? s_aoff[1] : 0u;
#pragma unroll 2
  for (int tt = 0; tt < gt; ++tt, blo += bstep) {
    const uint32_t off2 = tt + 2 < gt ? s_aoff[tt + 2] : 0u;    // two taps ahead
    uint32_t alo = hlo + off0;
    const uint32_t acc0 = (uint32_t)(!(first && tt == 0));
    if (MT == 1) {
#pragma unroll
      for (int k = 0; k < NK; ++k) umma_bf16_lh(tmem, alo + 2 * k, ahi, blo + 2 * k, bhi, idesc, k ? 1u : acc0);
    } else {
      for (int m = 0; m < MT; ++m, alo += a_mstep) {
        const uint32_t td = tmem + m * BN;
#pragma unroll
        for (int k = 0; k < NK; ++k) umma_bf16_lh(td, alo + 2 * k, ahi, blo + 2 * k, bhi, idesc, k ? 1u : acc0);
      }
    }
    off0 = off1;
    off1 = off2;
  }
}

template <int BN>
__global__ void __launch_bounds__(HaloCfg<BN>::kThreads, HaloCfg<BN>::kMinCtas) conv_halo_kernel(const __grid_constant__ CisConv p, const int halo_stage_bytes, const int BS, const int NHS,
                                                        const __grid_constant__ HaloMaps maps, const int use_tma, const int G) {
  // One weight pipeline stage = the tiles of G consecutive taps of one 64-channel chunk (contiguous in the pre-tiled operand, ONE
  // bulk copy): the single MMA-issuing thread then pays the per-stage cost (mbarrier wait, tcgen05 fence, election, commits: several
  // hundred clocks of dependent single-thread latency, measured with the CIS_TRACE build) once per 4*MT*G MMAs instead of once per
  // 4*MT -- that cost, not the tensor pipe, bounded every launch of round 1.
  // Compact thin halo (p.thin): 8-channel planes of 16 B per pixel, one K=16 MMA per "tap" entry, BN x 32 B weight tiles.
  const int thin = p.thin;
  const int kBStage = thin ? BN * 32 : BN * 128;
  constexpr int kHMmaWarp_ = HaloCfg<BN>::kMmaWarp, kHThreads_ = HaloCfg<BN>::kThreads;
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bars[2 * 2 + 2 * kHaloMaxBStages + 1];
  __shared__ uint32_t tmem_slot;
  __shared__ uint32_t s_aoff[CIS_MAX_TAPS];   // tap origin inside the halo, in descriptor start-field units (16 B)
  __shared__ SrcS s_src[CIS_MAX_SRC];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int MT = p.MT, d = p.dil;
  const int nph = p.nph > 1 ? p.nph : 1;       // stride-2 forward conv: 4 space-to-depth phases, each with its own halo and tap range
  const int Wh = 8 + p.ex, Hh = 16 * MT + p.ey, HP = Wh * Hh;
  const uint32_t stage_bytes = (uint32_t)G * kBStage;
  const uint32_t tile_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t h_base = tile_base;                                // NHS halo stages
  const uint32_t b_base = tile_base + NHS * halo_stage_bytes;       // BS weight stages of G tap tiles each
  int* pixtab = reinterpret_cast<int*>(smem_raw + (b_base + BS * stage_bytes - smem_u32(smem_raw)));
  const uint32_t bar_hfull = smem_u32(&bars[0]), bar_hempty = smem_u32(&bars[2]);
  const uint32_t bar_bfull = smem_u32(&bars[4]), bar_bempty = smem_u32(&bars[4 + kHaloMaxBStages]);
  const uint32_t bar_accum = smem_u32(&bars[4 + 2 * kHaloMaxBStages]);

  // ---- grouped launch: blockIdx.z selects one of nsub sub-problems (own taps, halo origin, weights, output extent / offset)
  const bool grouped = p.nsub > 1;
  const int tap0 = grouped ? p.sub[blockIdx.z].tap0 : 0, ntaps = grouped ? p.sub[blockIdx.z].ntaps : p.ntaps;
  const int hoy = grouped ? p.sub[blockIdx.z].hoy : p.hoy, hox = grouped ? p.sub[blockIdx.z].hox : p.hox;
  const int OHs = grouped ? p.sub[blockIdx.z].OH : p.OH, OWs = grouped ? p.sub[blockIdx.z].OW : p.OW;
  const int oa = grouped ? p.sub[blockIdx.z].oa : p.oa, ob = grouped ? p.sub[blockIdx.z].ob : p.ob;
  const void* const wpack = grouped ? p.sub[blockIdx.z].wpack : p.wpack;
  // ---- tile decode: blockIdx.x -> (tx, ty, phase, n)
  const int Hp0 = (OHs + d - 1) / d, Wp0 = (OWs + d - 1) / d;
  const int tiles_x = (Wp0 + 7) / 8, tiles_y = (Hp0 + 16 * MT - 1) / (16 * MT);
  if (grouped && (int)blockIdx.x >= tiles_x * tiles_y * p.N) return;   // the grid is sized for the largest sub-problem (uniform per CTA)
  int bid = blockIdx.x;
  const int tx = bid % tiles_x; bid /= tiles_x;
  const int ty = bid % tiles_y; bid /= tiles_y;
  const int ph = bid % (d * d);
  const int n = bid / (d * d);
  const int pa = ph / d, pb = ph % d;
  const int ny = blockIdx.y;
  int m_chunks = 0;
  for (int i = 0; i < p.nsrc; ++i) m_chunks += p.src[i].chunks;
  const int nchunks_all = (m_chunks + 7) / 8;  // 64-channel chunks
  const int nsplit = (!grouped && p.splits > 1) ? p.splits : 1;
  const int cper = (nchunks_all + nsplit - 1) / nsplit;
  const int cc_lo = grouped ? 0 : blockIdx.z * cper;
  const int nchunks = min(cper, nchunks_all - cc_lo);   // chunks handled by this CTA (host guarantees >= 1)
  __shared__ __align__(16) float s_bias[BN];
  pdl_launch_dependents();
  const uint32_t ncols = (MT * BN <= 32) ? 32u : (MT * BN <= 64) ? 64u : (MT * BN <= 128) ? 128u : (MT * BN <= 256) ? 256u : 512u;

  if (tid < ntaps) s_aoff[tid] = (uint32_t)((p.dh[tap0 + tid] * Wh + p.dw[tap0 + tid]) * (thin ? 1 : 8));   // * pixel bytes / 16
  if (tid < p.nsrc) {
    s_src[tid].ptr = reinterpret_cast<const __nv_bfloat16*>(p.src[tid].ptr);
    s_src[tid].pitch = p.src[tid].pitch;
    s_src[tid].c_off = p.src[tid].c_off;
    s_src[tid].chunks = p.src[tid].chunks;
    s_src[tid].n_mod = p.src[tid].n_mod;
  }
  for (int q = tid; q < (use_tma ? 0 : HP); q += kHThreads_) {
    const int hy = q / Wh, hx = q - hy * Wh;
    const int gy = ty * 16 * MT + hy + hoy, gx = tx * 8 + hx + hox;
    const int y = pa + d * gy, x = pb + d * gx;
    pixtab[q] = (gy >= 0 && gx >= 0 && y < p.H && x < p.W) ? (y * p.W + x) : -1;
  }
  if (warp == kHMmaWarp_) {
    if (lane == 0) {
      for (int s = 0; s < 2; ++s) {
        mbar_init(bar_hfull + 8 * s, use_tma ? 1 : 96);
        mbar_init(bar_hempty + 8 * s, 1);
      }
      for (int s = 0; s < BS; ++s) {
        mbar_init(bar_bfull + 8 * s, 1);   // one expect_tx arrival; the bulk copy completes the transaction bytes
        mbar_init(bar_bempty + 8 * s, 1);  // one commit by the MMA thread
      }
      mbar_init(bar_accum, 1);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc_dyn(smem_u32(&tmem_slot), ncols);
  }
  if (use_tma && tid < p.nsrc) tma_prefetch_desc(&maps.m[tid]);   // descriptors live in the kernel parameters: fetch them before the grid dependency resolves
  pdl_wait();
  if (tid < BN) s_bias[tid] = p.bias ? p.bias[ny * BN + tid] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  if (tid == 0) CIS_TRACE_AT(0);

  if (warp < kHMmaWarp_) {
   if (warp < 4) {
    // ------------------------------------------------------------------ producers
    // Two independent roles so neither stream throttles the other: warps 0-1 stream the per-chunk halos (2 stages), warps 2-3
    // stream the per-(tap, chunk) weight tiles (BS stages).
    if (use_tma) {
      if (tid == 0) {
        // halo through the TMA engine: one 4-D tiled load per 64-channel chunk (x phase), out-of-image pixels / channels are zero-filled
        int hcount = 0;
        for (int vc = 0; vc < nchunks * nph; ++vc) {
          const int cc = vc / nph, ph = vc - cc * nph;
          if (nph > 1 && p.ph_tap[ph + 1] == p.ph_tap[ph]) continue;      // phase without taps (kernel size 1)
          const int hs = hcount % NHS;
          mbar_wait(bar_hempty + 8 * hs, (uint32_t)(((hcount / NHS) & 1) ^ 1));
          ++hcount;
          int c = (cc_lo + cc) * 8, si = 0;
          while (si < p.nsrc - 1 && c >= s_src[si].chunks) {
            c -= s_src[si].chunks;
            ++si;
          }
          if (thin) {
            // one 16-byte-per-pixel plane per 8-channel chunk of the (<= 16-channel) concat
            const uint32_t plane = thin_plane_bytes(HP);
            mbar_expect_tx(bar_hfull + 8 * hs, (uint32_t)(m_chunks * HP * 16));
            for (int q = 0; q < m_chunks; ++q) {       // <= 2 planes: source 0, or sources 0 and 1 with one chunk each
              const int sq = q < s_src[0].chunks ? 0 : 1, cq = q - (sq ? s_src[0].chunks : 0);
              const int nm = s_src[sq].n_mod;
              tma_load_4d(h_base + hs * halo_stage_bytes + q * plane, &maps.m[sq * nph + ph], bar_hfull + 8 * hs, cq * 8, tx * 8 + hox,
                          ty * 16 * MT + hoy, nm ? (n % nm) : n);
            }
            continue;
          }
          const int nmod = s_src[si].n_mod;
          mbar_expect_tx(bar_hfull + 8 * hs, (uint32_t)(HP * 128));
          // dilated layer: the map strides by d pixels from any start, the start carries this CTA's phase (pa, pb)
          tma_load_4d(h_base + hs * halo_stage_bytes, &maps.m[si * nph + ph], bar_hfull + 8 * hs, c * 8, pb + d * (tx * 8 + hox),
                      pa + d * (ty * 16 * MT + hoy), nmod ? (n % nmod) : n);
        }
      }
      __syncwarp();
    } else if (warp != 2) {
      const int hid = warp == 3 ? tid - 32 : tid;   // 96 halo loader threads (warps 0, 1, 3)
      const int j = hid & 7, pl = hid >> 3;         // pl = 0..11
      for (int cc = 0; cc < nchunks; ++cc) {
        const int hs = cc % NHS;
        mbar_wait(bar_hempty + 8 * hs, (uint32_t)(((cc / NHS) & 1) ^ 1));
        const int rem = m_chunks - (cc_lo + cc) * 8;       // valid 16-byte chunks in this 64-channel chunk
        const int nk16 = rem >= 8 ? 4 : (rem + 1) / 2;     // K=16 MMA groups actually issued
        const bool need = j < 2 * nk16;
        const bool cvalid = j < rem;
        int c = (cc_lo + cc) * 8 + j, si = 0;
        if (cvalid) {
          while (si < p.nsrc - 1 && c >= s_src[si].chunks) {
            c -= s_src[si].chunks;
            ++si;
          }
        } else {
          c = 0;
        }
        const int nmod = s_src[si].n_mod, pitch = s_src[si].pitch;
        const int ne = nmod ? (n % nmod) : n;
        const __nv_bfloat16* sp = s_src[si].ptr;
        const __nv_bfloat16* sb = sp + (size_t)ne * p.H * p.W * pitch + s_src[si].c_off + c * 8;
        if (need) {
          const uint32_t hdst = h_base + hs * halo_stage_bytes + (uint32_t)(j << 4);
          for (int q = pl; q < HP; q += 12) {
            const int off = pixtab[q];
            const bool ok = cvalid && off >= 0;
            cp_async16((hdst + q * 128) ^ (uint32_t)((q & 7) << 4), ok ? (const void*)(sb + (size_t)off * pitch) : (const void*)sp,
                       ok ? 16u : 0u);
          }
        }
        cp_async_commit();
        if (NHS == 1) {
          cp_async_wait<0>();
          fence_proxy_async();
          mbar_arrive(bar_hfull);
        } else if (cc >= 1) {        // two stages: publish chunk cc-1 while chunk cc is in flight
          cp_async_wait<1>();
          fence_proxy_async();
          mbar_arrive(bar_hfull + 8 * ((cc - 1) % NHS));
        }
      }
      if (NHS > 1) {
        cp_async_wait<0>();
        fence_proxy_async();
        mbar_arrive(bar_hfull + 8 * ((nchunks - 1) % NHS));
      }
    }
    if (tid == 64) {
      // weights: pre-swizzled [n-tile][chunk][tap] tiles of BN x 128 B (cis_pack_weights_tiled); the tiles of the G taps of a stage
      // are adjacent in that layout -> ONE bulk copy per pipeline stage
      const uint8_t* wt = reinterpret_cast<const uint8_t*>(wpack) + ((size_t)ny * nchunks_all + cc_lo) * ntaps * kBStage;
      int bs = 0;
      uint32_t bph = 1;           // parity to wait for on the empty barrier: the first pass over the ring finds every stage free
      for (int vc = 0; vc < nchunks * nph; ++vc) {
        const int cc = vc / nph, ph = vc - cc * nph;
        const int tlo = nph > 1 ? p.ph_tap[ph] : 0, thi = nph > 1 ? p.ph_tap[ph + 1] : ntaps;
        for (int t0 = tlo; t0 < thi; t0 += G) {
          const uint32_t bytes = (uint32_t)min(G, thi - t0) * kBStage;
          mbar_wait(bar_bempty + 8 * bs, bph);
          mbar_expect_tx(bar_bfull + 8 * bs, bytes);
          bulk_g2s(b_base + bs * stage_bytes, wt + (size_t)(cc * ntaps + t0) * kBStage, bytes, bar_bfull + 8 * bs);
          if (++bs == BS) {
            bs = 0;
            bph ^= 1u;
          }
        }
      }
    }
    __syncwarp();
   }

    // ------------------------------------------------------------------ epilogue: warps w and w + 4 share TMEM lane quarter w % 4 and
    // split the columns (the epilogue is instruction-bound on its warps: ~6k clk per 128x128 tile with four of them, r02 trace)
    mbar_wait(bar_accum, 0);
    tc_fence_after();
    if (tid == 0) CIS_TRACE_AT(2);
    const int qtr = warp & 3, half = warp >> 2;
    const int r = qtr * 32 + lane;
    const int c_lo = (kHMmaWarp_ == 8) ? half * (BN / 2) : 0, c_hi = (kHMmaWarp_ == 8) ? c_lo + BN / 2 : BN;
    const uint32_t t_qtr = tmem + ((uint32_t)(qtr * 32) << 16);
    const int cbase = ny * BN;
    const int tile_id = blockIdx.x * gridDim.y + ny;
    if (nsplit > 1 && p.sk_cluster) {
      // cluster split-K: the MT partial tiles -> own shared memory (operand buffers are dead: every MMA has completed); reduced below
      for (int m = 0; m < MT; ++m)
        if (c_lo < c_hi) tmem_to_stage(t_qtr + m * BN, r, tile_base + (uint32_t)m * (kBM * BN * 4), c_lo, c_hi);
    } else if (nsplit > 1) {
      // two-launch split-K: this split's private fp32 slices; splitk_finish_kernel reduces them and runs the fused epilogue
      for (int m = 0; m < MT; ++m)
        if (c_lo < c_hi)
          splitk_store_partial<BN>(p.sk_scratch + (((size_t)tile_id * MT + m) * nsplit + blockIdx.z) * kBM * BN, t_qtr + m * BN, r, c_lo, c_hi);
    } else if (c_lo < c_hi) {
      for (int m = 0; m < MT; ++m) {
        const int gy = ty * 16 * MT + 16 * m + (r >> 3), gx = tx * 8 + (r & 7);
        const int oy = pa + d * gy, ox = pb + d * gx;
        const bool valid = oy < OHs && ox < OWs;
        const size_t dpix = valid ? ((size_t)(n * p.DH + oy * p.osh + oa) * p.DW + ox * p.osw + ob) : 0;
        epi_cols<BN>(p, t_qtr + m * BN, cbase, dpix, valid, s_bias, c_lo, c_hi);
      }
    }
  } else {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = make_idesc_bf16(kBM, BN, 0, 0);
    // compact halo: SWIZZLE_NONE, SBO = one halo row; the second K half of an MMA is the next pixel (8 channels: x-adjacent tap,
    // LBO = 16 B) or the next plane (16 channels); weights [K half][BN][16 B] (LBO = BN x 16 B, SBO = 128 B)
    const uint32_t ahi = thin ? desc_hi_noswz((uint32_t)(Wh * 16)) : desc_hi((uint32_t)(Wh * 128));
    const uint32_t bhi = thin ? desc_hi_noswz(128u) : desc_hi(1024);
    const uint32_t a_lbo = thin ? (m_chunks == 1 ? 16u : thin_plane_bytes(HP)) : 16u, b_lbo = thin ? (uint32_t)(BN * 16) : 16u;
    const uint32_t a_mstep = (uint32_t)(16 * Wh * (thin ? 16 : 128)) >> 4;   // descriptor start-field step between stacked M tiles
    const uint32_t bstep = (uint32_t)kBStage >> 4;
    int bs = 0, hs = 0, it = 0;
    uint32_t bph = 0, hph = 0;
    int vlast = nchunks * nph - 1;                       // last virtual chunk that has taps
    while (nph > 1 && vlast > 0 && p.ph_tap[vlast % nph + 1] == p.ph_tap[vlast % nph]) --vlast;
    bool any = false;
    for (int vc = 0; vc < nchunks * nph; ++vc) {
      const int cc = vc / nph, ph = vc - cc * nph;
      const int tlo = nph > 1 ? p.ph_tap[ph] : 0, thi = nph > 1 ? p.ph_tap[ph + 1] : ntaps;
      if (thi == tlo) continue;
      const int rem = m_chunks - (cc_lo + cc) * 8;
      const int nk16 = rem >= 8 ? 4 : (rem + 1) / 2;
      mbar_wait(bar_hfull + 8 * hs, hph);
      if (vc == 0 && lane == 0) CIS_TRACE_AT(1);
      const uint32_t hlo = desc_lo(h_base + hs * halo_stage_bytes, a_lbo);
      for (int t0 = tlo; t0 < thi; t0 += G, ++it) {
        const int gt = min(G, thi - t0);
        mbar_wait(bar_bfull + 8 * bs, bph);
        tc_fence_after();
        if (elect_one()) {
          CIS_TRACE_AT(8 + 2 * it);
          const uint32_t blo = desc_lo(b_base + bs * stage_bytes, b_lbo);
          const bool first = !any;
          if (nk16 == 4) halo_issue_stage<4>(tmem, hlo, blo, s_aoff + t0, gt, MT, BN, ahi, bhi, a_mstep, bstep, idesc, first);
          else if (nk16 == 1) halo_issue_stage<1>(tmem, hlo, blo, s_aoff + t0, gt, MT, BN, ahi, bhi, a_mstep, bstep, idesc, first);
          else if (nk16 == 2) halo_issue_stage<2>(tmem, hlo, blo, s_aoff + t0, gt, MT, BN, ahi, bhi, a_mstep, bstep, idesc, first);
          else halo_issue_stage<3>(tmem, hlo, blo, s_aoff + t0, gt, MT, BN, ahi, bhi, a_mstep, bstep, idesc, first);
          umma_commit(bar_bempty + 8 * bs);
          if (t0 + G >= thi) {
            umma_commit(bar_hempty + 8 * hs);
            if (vc == vlast) umma_commit(bar_accum);
          }
          CIS_TRACE_AT(9 + 2 * it);
        }
        __syncwarp();
        any = true;
        if (++bs == BS) {
          bs = 0;
          bph ^= 1u;
        }
      }
      if (++hs == NHS) {
        hs = 0;
        hph ^= 1u;
      }
    }
  }
  if (nsplit > 1 && p.sk_cluster) {
    cluster_sync_all();                       // every CTA's partial tiles are in its shared memory
    if (warp < 4) {
      const int cbase = ny * BN;
      for (int m = 0; m < MT; ++m)
        cluster_reduce_rows<BN>(p, tile_base + (uint32_t)m * (kBM * BN * 4), nsplit, (int)cluster_ctarank(), tid, 128, cbase,
                                [&](int row, bool& valid) -> size_t {
                                  const int gy = ty * 16 * MT + 16 * m + (row >> 3), gx = tx * 8 + (row & 7);
                                  const int oy = pa + d * gy, ox = pb + d * gx;
                                  valid = oy < OHs && ox < OWs;
                                  return valid ? ((size_t)(n * p.DH + oy * p.osh + oa) * p.DW + ox * p.osw + ob) : 0;
                                });
    }
    cluster_sync_all();                       // peers may still be reading this CTA's shared memory
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0) CIS_TRACE_AT(3);
  if (warp == kHMmaWarp_) tmem_dealloc_dyn(tmem, ncols);
}

// ======================================================================================================= split-K finish
// Second launch of split-K.  (Round 1 let the last-arriving CTA of a tile read all nsplit x 64 KB slices by itself -- one SM pulling up
// to 1 MB through L2 -- which cost more than the split saved on the low-resolution layers it is meant for.)  Here the reduction + fused
// epilogue of a tile is spread over 128 * BN/16 threads of several CTAs: thread = (accumulator row, 16-column group), row fastest so
// the reads of the float4-column slices coalesce (the bf16 output is 1 / (2 * nsplit) of the bytes: its 32-byte pieces matter less).
template <int BN>
__global__ void __launch_bounds__(256) splitk_finish_kernel(const __grid_constant__ CisConv p) {
  constexpr int G = BN / 16;                               // 16-column groups per row
  constexpr int kBlock = (128 * G < 256) ? 128 * G : 256;
  constexpr int kSub = 128 * G / kBlock;                   // CTAs per (tile, m)
  pdl_launch_dependents();
  pdl_wait();
  const int tid = threadIdx.x;
  if (tid >= kBlock) return;
  const int m = blockIdx.z / kSub;
  const int item = (blockIdx.z % kSub) * kBlock + tid;
  const int r = item % 128, c0 = (item / 128) * 16;        // row fastest: a warp reads 512 contiguous bytes of every slice
  const int ny = blockIdx.y;
  const int nsplit = p.splits;
  const int tile_id = blockIdx.x * gridDim.y + ny;
  bool valid;
  size_t dpix = 0;
  const float* tile0;
  if (p.halo) {
    const int MT = p.MT, d = p.dil;
    const int Hp0 = (p.OH + d - 1) / d, Wp0 = (p.OW + d - 1) / d;
    const int tiles_x = (Wp0 + 7) / 8, tiles_y = (Hp0 + 16 * MT - 1) / (16 * MT);
    int bid = blockIdx.x;
    const int tx = bid % tiles_x; bid /= tiles_x;
    const int ty = bid % tiles_y; bid /= tiles_y;
    const int ph = bid % (d * d);
    const int n = bid / (d * d);
    const int pa = ph / d, pb = ph % d;
    const int gy = ty * 16 * MT + 16 * m + (r >> 3), gx = tx * 8 + (r & 7);
    const int oy = pa + d * gy, ox = pb + d * gx;
    valid = oy < p.OH && ox < p.OW;
    if (valid) dpix = (size_t)(n * p.DH + oy * p.osh + p.oa) * p.DW + ox * p.osw + p.ob;
    tile0 = p.sk_scratch + ((size_t)tile_id * MT + m) * nsplit * kBM * BN;
  } else {
    const int M = p.N * p.OH * p.OW;
    const int g = blockIdx.x * kBM + r;
    valid = g < M;
    if (valid) {
      const int ow = g % p.OW;
      const int t = g / p.OW;
      const int oh = t % p.OH;
      const int n = t / p.OH;
      dpix = (size_t)(n * p.DH + oh * p.osh + p.oa) * p.DW + ow * p.osw + p.ob;
    }
    tile0 = p.sk_scratch + (size_t)tile_id * nsplit * kBM * BN;
  }
  if (!valid) return;
  float v[16];
  splitk_reduce16<BN>(tile0, nsplit, r, c0, v);
  epi_chunk(p, v, ny * BN + c0, dpix);
}
// ======================================================================================================= persistent halo conv
// Same math as conv_halo_kernel (TMA halo path only) for layers with MANY output tiles per SM (high-resolution thin layers), where the
// per-CTA prologue (barrier init, TMEM allocation, first TMA round trip: ~3k clk) and epilogue (TMEM read-back + stores on one warp
// per scheduler: 2-17k clk) of the one-tile-per-CTA kernel cost more than its MMA loop (CIS_TRACE build, r02).  Here a CTA is
// persistent and fully warp-specialised so those phases of neighbouring tiles overlap:
//   warp 0: halo TMA producer (NHS stages) | warp 1: weight producer | warp 2: MMA issuer | warp 3: TMEM owner
//   warps 4-7 / 8-11: two epilogue groups (TMEM lane quarter = warp % 4); tile i uses accumulator stage i % AS and group i % AS.
// Weights: resident (ws = 1: the whole set of nchunks*ntaps tiles is fetched once per CTA and stays in shared memory while the CTA
// walks its tiles) when it fits, else re-streamed per tile in stages of G taps through a ring of BS stages.
// Every role walks the same static work list  w = blockIdx.x, blockIdx.x + gridDim.x, ...  of output tiles.
static constexpr int kPThreads = 384;

template <int BN>
__global__ void __launch_bounds__(kPThreads, 2) conv_halo_persist_kernel(const __grid_constant__ CisConv p, const int halo_stage_bytes,
                                                                       const int BS, const int NHS, const int AS, const int G,
                                                                       const __grid_constant__ HaloMaps maps, const int ws) {
  const int thin = p.thin;                       // compact thin halo: see conv_halo_kernel
  const int kBStage = thin ? BN * 32 : BN * 128;
  constexpr int kMaxHS = 4;
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bars[2 * kMaxHS + 2 * kHaloMaxBStages + 4];
  __shared__ uint32_t tmem_slot;
  __shared__ uint32_t s_aoff[CIS_MAX_TAPS];
  __shared__ __align__(16) float s_bias[BN];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int MT = p.MT;
  const int Wh = 8 + p.ex, Hh = 16 * MT + p.ey, HP = Wh * Hh;
  const uint32_t stage_bytes = (uint32_t)G * kBStage;
  const uint32_t tile_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t h_base = tile_base, b_base = tile_base + NHS * halo_stage_bytes;
  const uint32_t bar_hfull = smem_u32(&bars[0]), bar_hempty = smem_u32(&bars[kMaxHS]);
  const uint32_t bar_bfull = smem_u32(&bars[2 * kMaxHS]), bar_bempty = smem_u32(&bars[2 * kMaxHS + kHaloMaxBStages]);
  const uint32_t bar_tfull = smem_u32(&bars[2 * kMaxHS + 2 * kHaloMaxBStages]), bar_tempty = smem_u32(&bars[2 * kMaxHS + 2 * kHaloMaxBStages + 2]);

  const int tiles_x = (p.OW + 7) / 8, tiles_y = (p.OH + 16 * MT - 1) / (16 * MT);
  const int total = tiles_x * tiles_y * p.N;
  int m_chunks = 0;
  for (int i = 0; i < p.nsrc; ++i) m_chunks += p.src[i].chunks;
  const int nchunks = (m_chunks + 7) / 8;
  const uint32_t acc_cols = (uint32_t)(MT * BN);
  const uint32_t want = acc_cols * AS;
  const uint32_t ncols = want <= 32 ? 32u : want <= 64 ? 64u : want <= 128 ? 128u : want <= 256 ? 256u : 512u;

  pdl_launch_dependents();
  if (tid < p.ntaps) s_aoff[tid] = (uint32_t)((p.dh[tid] * Wh + p.dw[tid]) * (thin ? 1 : 8));
  if (warp == 3) {
    if (lane == 0) {
      for (int s = 0; s < NHS; ++s) {
        mbar_init(bar_hfull + 8 * s, 1);
        mbar_init(bar_hempty + 8 * s, 1);
      }
      for (int s = 0; s < BS; ++s) {
        mbar_init(bar_bfull + 8 * s, 1);
        mbar_init(bar_bempty + 8 * s, 1);
      }
      for (int s = 0; s < AS; ++s) {
        mbar_init(bar_tfull + 8 * s, 1);
        mbar_init(bar_tempty + 8 * s, 4);   // one arrival per warp of the epilogue group that drained the stage
      }
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc_dyn(smem_u32(&tmem_slot), ncols);
  }
  if (tid < p.nsrc) tma_prefetch_desc(&maps.m[tid]);
  pdl_wait();
  if (tid < BN) s_bias[tid] = p.bias ? p.bias[tid] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  if (tid == 0) {
    CIS_TRACE_AT(0);
    CIS_TRACE_AT(4);      // slot 4 marks a persistent-kernel trace (tools/trace_persist.py)
  }

  if (warp == 0) {
    // ------------------------------------------------------------------ halo producer
    if (lane == 0) {
      int hs = 0;
      uint32_t hph = 1;
      for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const int tx = w % tiles_x, r1 = w / tiles_x, ty = r1 % tiles_y, n = r1 / tiles_y;
        for (int cc = 0; cc < nchunks; ++cc) {
          mbar_wait(bar_hempty + 8 * hs, hph);
          int c = cc * 8, si = 0;
          while (si < p.nsrc - 1 && c >= p.src[si].chunks) {
            c -= p.src[si].chunks;
            ++si;
          }
          if (thin) {
            const uint32_t plane = thin_plane_bytes(HP);
            mbar_expect_tx(bar_hfull + 8 * hs, (uint32_t)(m_chunks * HP * 16));
            for (int q = 0; q < m_chunks; ++q) {       // <= 2 planes: source 0, or sources 0 and 1 with one chunk each
              const int sq = q < p.src[0].chunks ? 0 : 1, cq = q - (sq ? p.src[0].chunks : 0);
              const int nm = sq ? p.src[1].n_mod : p.src[0].n_mod;
              tma_load_4d(h_base + hs * halo_stage_bytes + q * plane, &maps.m[sq], bar_hfull + 8 * hs, cq * 8, tx * 8 + p.hox,
                          ty * 16 * MT + p.hoy, nm ? (n % nm) : n);
            }
          } else {
            int nmod = p.src[0].n_mod;
            if (si == 1) nmod = p.src[1].n_mod;
            if (si == 2) nmod = p.src[2].n_mod;
            if (si == 3) nmod = p.src[3].n_mod;
            mbar_expect_tx(bar_hfull + 8 * hs, (uint32_t)(HP * 128));
            tma_load_4d(h_base + hs * halo_stage_bytes, &maps.m[si], bar_hfull + 8 * hs, c * 8, tx * 8 + p.hox, ty * 16 * MT + p.hoy,
                        nmod ? (n % nmod) : n);
          }
          if (++hs == NHS) {
            hs = 0;
            hph ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ weight producer
    if (lane == 0) {
      const uint8_t* wt = reinterpret_cast<const uint8_t*>(p.wpack);
      const int per_tile = nchunks * p.ntaps;
      if (ws) {
        if ((int)blockIdx.x < total) {
          mbar_expect_tx(bar_bfull, (uint32_t)(per_tile * kBStage));
          for (int it = 0; it < per_tile; it += 8) {      // bulk copies of up to 8 tiles (<= 128 KB each)
            const int nt = min(8, per_tile - it);
            bulk_g2s(b_base + it * kBStage, wt + (size_t)it * kBStage, (uint32_t)(nt * kBStage), bar_bfull);
          }
        }
      } else {
        int bs = 0;
        uint32_t bph = 1;
        for (int w = blockIdx.x; w < total; w += gridDim.x) {
          for (int cc = 0; cc < nchunks; ++cc) {
            for (int t0 = 0; t0 < p.ntaps; t0 += G) {
              const uint32_t bytes = (uint32_t)min(G, p.ntaps - t0) * kBStage;
              mbar_wait(bar_bempty + 8 * bs, bph);
              mbar_expect_tx(bar_bfull + 8 * bs, bytes);
              bulk_g2s(b_base + bs * stage_bytes, wt + (size_t)(cc * p.ntaps + t0) * kBStage, bytes, bar_bfull + 8 * bs);
              if (++bs == BS) {
                bs = 0;
                bph ^= 1u;
              }
            }
          }
        }
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = make_idesc_bf16(kBM, BN, 0, 0);
    const uint32_t ahi = thin ? desc_hi_noswz((uint32_t)(Wh * 16)) : desc_hi((uint32_t)(Wh * 128));
    const uint32_t bhi = thin ? desc_hi_noswz(128u) : desc_hi(1024);
    const uint32_t a_lbo = thin ? (m_chunks == 1 ? 16u : thin_plane_bytes(HP)) : 16u, b_lbo = thin ? (uint32_t)(BN * 16) : 16u;
    const uint32_t a_mstep = (uint32_t)(16 * Wh * (thin ? 16 : 128)) >> 4;
    const uint32_t bstep = (uint32_t)kBStage >> 4;
    int hs = 0, bs = 0, as = 0;
    uint32_t hph = 0, bph = 0, tph = 1;
    if (ws && (int)blockIdx.x < total) {
      mbar_wait(bar_bfull, 0u);      // the resident weight set; never released
      tc_fence_after();
    }
    int wi = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x, ++wi) {
      if (lane == 0) CIS_TRACE_AT(8 + 5 * wi);
      mbar_wait(bar_tempty + 8 * as, tph);
      tc_fence_after();
      if (lane == 0) CIS_TRACE_AT(9 + 5 * wi);
      const uint32_t tacc = tmem + as * acc_cols;
      for (int cc = 0; cc < nchunks; ++cc) {
        const int rem = m_chunks - cc * 8;
        const int nk16 = rem >= 8 ? 4 : (rem + 1) / 2;
        mbar_wait(bar_hfull + 8 * hs, hph);
        if (cc == 0 && lane == 0) CIS_TRACE_AT(10 + 5 * wi);
        const uint32_t hlo = desc_lo(h_base + hs * halo_stage_bytes, a_lbo);
        const int gstep = ws ? p.ntaps : G;
        for (int t0 = 0; t0 < p.ntaps; t0 += gstep) {
          const int gt = min(gstep, p.ntaps - t0);
          if (!ws) mbar_wait(bar_bfull + 8 * bs, bph);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t blo = desc_lo(ws ? b_base + (uint32_t)(cc * p.ntaps) * kBStage : b_base + bs * stage_bytes, b_lbo);
            const bool first = (cc | t0) == 0;
            if (nk16 == 4) halo_issue_stage<4>(tacc, hlo, blo, s_aoff + t0, gt, MT, BN, ahi, bhi, a_mstep, bstep, idesc, first);
            else if (nk16 == 1) halo_issue_stage<1>(tacc, hlo, blo, s_aoff + t0, gt, MT, BN, ahi, bhi, a_mstep, bstep, idesc, first);
            else if (nk16 == 2) halo_issue_stage<2>(tacc, hlo, blo, s_aoff + t0, gt, MT, BN, ahi, bhi, a_mstep, bstep, idesc, first);
            else halo_issue_stage<3>(tacc, hlo, blo, s_aoff + t0, gt, MT, BN, ahi, bhi, a_mstep, bstep, idesc, first);
            if (!ws) umma_commit(bar_bempty + 8 * bs);
            if (t0 + gstep >= p.ntaps) {
              umma_commit(bar_hempty + 8 * hs);
              if (cc == nchunks - 1) {
                umma_commit(bar_tfull + 8 * as);
                CIS_TRACE_AT(11 + 5 * wi);
              }
            }
          }
          __syncwarp();
          if (!ws && ++bs == BS) {
            bs = 0;
            bph ^= 1u;
          }
        }
        if (++hs == NHS) {
          hs = 0;
          hph ^= 1u;
        }
      }
      if (++as == AS) {
        as = 0;
        tph ^= 1u;
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue: group g = (warp - 4) / 4 drains accumulator stage g
    const int grp = (warp - 4) >> 2, q = warp & 3;
    const int r = q * 32 + lane;
    if (grp < AS) {
      uint32_t tph = 0;
      int wi = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x, ++wi) {
        if (wi % AS != grp) continue;
        const int tx = w % tiles_x, r1 = w / tiles_x, ty = r1 % tiles_y, n = r1 / tiles_y;
        mbar_wait(bar_tfull + 8 * grp, tph);
        tph ^= 1u;
        tc_fence_after();
        for (int m = 0; m < MT; ++m) {
          const int oy = ty * 16 * MT + 16 * m + (r >> 3), ox = tx * 8 + (r & 7);
          const bool valid = oy < p.OH && ox < p.OW;
          const size_t dpix = valid ? ((size_t)(n * p.DH + oy * p.osh + p.oa) * p.DW + ox * p.osw + p.ob) : 0;
          epi_row<BN>(p, tmem + ((uint32_t)(q * 32) << 16) + grp * acc_cols + m * BN, 0, dpix, valid, s_bias);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_tempty + 8 * grp);
        if (q == 0 && lane == 0) CIS_TRACE_AT(12 + 5 * wi);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 3) tmem_dealloc_dyn(tmem, ncols);
}

// ======================================================================================================= wgrad
// D[co][kcol] = sum_pix g[pix][co] * A[pix][kcol]; both operands are "MN-major" (the reduction dim = pixels is the slow
// dimension of NHWC), staged as two [64 pixels][64 channels] SWIZZLE_128B sub-tiles each.
static constexpr int kWStages = 3;
static constexpr int kWTile = 64 * 128;            // one [64 pix][64 ch] bf16 sub-tile
static constexpr int kWStage = 4 * kWTile;         // A (2 sub-tiles) + B (2 sub-tiles)
static constexpr int kWSmem = kWStages * kWStage + 1024;

struct WgradMaps {
  CUtensorMap g;                 // (C8, OW, OH, N) gradient slice, box (64, 8, 8, 1)
  CUtensorMap x[CIS_MAX_SRC];    // (C8, W, H, N) activation slices, box (64, 8, 8, 1)
};

__global__ void __launch_bounds__(kGThreads) conv_wgrad_kernel(const __grid_constant__ CisWgrad p, const __grid_constant__ WgradMaps maps) {
  constexpr int S = kWStages;
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bars[2 * S + 1];
  __shared__ uint32_t tmem_slot;
  __shared__ int s_dh[CIS_MAX_TAPS], s_dw[CIS_MAX_TAPS];
  const uint32_t tile_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = smem_u32(&bars[0]);
  const uint32_t bar_empty = smem_u32(&bars[S]);
  const uint32_t bar_accum = smem_u32(&bars[2 * S]);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // blockDim = producer/epilogue warps + 1 MMA warp: 4 + 1 on the TMA operand path (one thread issues the loads), 8 + 1 on the
  // cp.async gather path, whose address arithmetic is the bottleneck (thin or strided layers)
  const int nprod = (int)blockDim.x - 32, mma_warp = nprod >> 5;
  pdl_launch_dependents();
  if (tid < p.ntaps) {
    s_dh[tid] = p.dh[tid];
    s_dw[tid] = p.dw[tid];
  }
  const int M = p.N * p.OH * p.OW;  // reduction length (pixels)
  int m_chunks = 0;
  for (int i = 0; i < p.nsrc; ++i) m_chunks += p.src[i].chunks;
  const int k_chunks = p.ntaps * m_chunks;
  const int tiles_x = (p.OW + 7) / 8, tiles_y = (p.OH + 7) / 8;
  const int nkb_total = p.tma ? p.N * tiles_x * tiles_y : (M + 63) / 64;   // TMA path: one K block = one 8x8 pixel tile
  const int per = (nkb_total + p.splits - 1) / p.splits;
  const int kb0 = blockIdx.y * per;
  const int kb1 = min(kb0 + per, nkb_total);
  const int nkb = kb1 - kb0;
  if (nkb <= 0) return;  // never taken: cis_conv_wgrad rejects split counts that leave a split without work (its slice would be garbage)

  if (warp == mma_warp) {
    if (lane == 0) {
      for (int s = 0; s < S; ++s) {
        mbar_init(bar_full + 8 * s, p.tma ? 1 : nprod);
        mbar_init(bar_empty + 8 * s, 1);
      }
      mbar_init(bar_accum, 1);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc<128>(smem_u32(&tmem_slot));
  }
  pdl_wait();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;

  if (warp < mma_warp) {
    if (p.tma) {
      if (tid == 0) {
        // two 64-column groups of this CTA: group = tap * nchunks64 + chunk64 -> (tap offset, source map, channel offset)
        const int nch64 = (m_chunks + 7) / 8;
        int gsrc[2], gc0[2], gdh[2], gdw[2], gnm[2];
        bool gok[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int grp = blockIdx.x * 2 + u;
          gok[u] = grp < p.ntaps * nch64;
          const int t = gok[u] ? grp / nch64 : 0;
          int c = gok[u] ? (grp - t * nch64) * 8 : 0, si = 0;
          while (si < p.nsrc - 1 && c >= p.src[si].chunks) {
            c -= p.src[si].chunks;
            ++si;
          }
          gsrc[u] = si;
          gc0[u] = c * 8;
          gdh[u] = s_dh[t];
          gdw[u] = s_dw[t];
          int nm = p.src[0].n_mod;
          if (si == 1) nm = p.src[1].n_mod;
          if (si == 2) nm = p.src[2].n_mod;
          if (si == 3) nm = p.src[3].n_mod;
          gnm[u] = nm;
        }
        const int tpi = tiles_x * tiles_y;
        for (int it = 0; it < nkb; ++it) {
          const int s = it % S;
          mbar_wait(bar_empty + 8 * s, (uint32_t)(((it / S) & 1) ^ 1));
          const int kb = kb0 + it;
          const int n = kb / tpi, r = kb - n * tpi;
          const int ty = r / tiles_x, tx = r - ty * tiles_x;
          const uint32_t st = tile_base + s * kWStage, bar = bar_full + 8 * s;
          mbar_expect_tx(bar, 4 * kWTile);
          tma_load_4d(st, &maps.g, bar, 0, tx * 8, ty * 8, n);
          tma_load_4d(st + kWTile, &maps.g, bar, 64, tx * 8, ty * 8, n);          // channels >= extent: zero fill
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int ne = gnm[u] ? (n % gnm[u]) : n;
            // an invalid group (beyond the last tap) reads channel 1<<20 -> fully out of range -> zeros
            tma_load_4d(st + (2 + u) * kWTile, &maps.x[gsrc[u]], bar, gok[u] ? gc0[u] : (1 << 20), tx * 8 + gdw[u], ty * 8 + gdh[u], ne);
          }
        }
      }
      __syncwarp();
    } else {
    const int j = tid & 7, rl = tid >> 3;
    const uint32_t sw_off = (uint32_t)((j ^ (rl & 7)) << 4);
    // fixed per-thread decode of the two B (activation) chunks and two A (gradient) chunks
    const __nv_bfloat16* bptr[2];
    int bpitch[2], bcoff[2], bnmod[2], bdh[2], bdw[2];
    bool bvalid[2], avalid[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int q = blockIdx.x * 16 + u * 8 + j;
      bvalid[u] = q < k_chunks;
      int t = 0, c = 0;
      if (bvalid[u]) {
        t = q / m_chunks;
        c = q - t * m_chunks;
      }
      int si = 0;
      while (si < p.nsrc - 1 && c >= p.src[si].chunks) {
        c -= p.src[si].chunks;
        ++si;
      }
      // static unrolled select keeps p.src[] accesses at constant indices
      CisSrc sd = p.src[0];
      if (si == 1) sd = p.src[1];
      if (si == 2) sd = p.src[2];
      if (si == 3) sd = p.src[3];
      bptr[u] = reinterpret_cast<const __nv_bfloat16*>(sd.ptr);
      bpitch[u] = sd.pitch;
      bcoff[u] = sd.c_off + c * 8;
      bnmod[u] = sd.n_mod;
      bdh[u] = s_dh[t];
      bdw[u] = s_dw[t];
      avalid[u] = (u * 8 + j) < p.g_chunks;
    }
    const __nv_bfloat16* gp = reinterpret_cast<const __nv_bfloat16*>(p.g);

    for (int it = 0; it < nkb; ++it) {
      const int s = it % S;
      const uint32_t ph = (uint32_t)((it / S) & 1);
      mbar_wait(bar_empty + 8 * s, ph ^ 1u);
      const uint32_t st = tile_base + s * kWStage;
#pragma unroll
      for (int r = rl; r < 64; r += nprod >> 3) {
        const int g = (kb0 + it) * 64 + r;
        const bool rv = g < M;
        int n = 0, h0 = 0, w0 = 0;
        if (rv) {
          const int ow = g % p.OW;
          const int t = g / p.OW;
          h0 = (t % p.OH) * p.sh;
          n = t / p.OH;
          w0 = ow * p.sw;
        }
        const uint32_t dst = st + r * 128 + sw_off;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const bool ok = rv && avalid[u];
          const size_t off = ok ? ((size_t)g * p.g_pitch + p.g_coff + (u * 8 + j) * 8) : 0;
          cp_async16(dst + u * kWTile, gp + off, ok ? 16u : 0u);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int h = h0 + bdh[u], w = w0 + bdw[u];
          const bool ok = rv && bvalid[u] && (unsigned)h < (unsigned)p.H && (unsigned)w < (unsigned)p.W;
          const int ne = bnmod[u] ? (n % bnmod[u]) : n;
          const size_t off = ok ? ((size_t)((ne * p.H + h) * p.W + w) * bpitch[u] + bcoff[u]) : 0;
          cp_async16(dst + (2 + u) * kWTile, bptr[u] + off, ok ? 16u : 0u);
        }
      }
      cp_async_commit();
      if (it >= S - 1) {
        cp_async_wait<S - 1>();
        fence_proxy_async();
        mbar_arrive(bar_full + 8 * ((it - (S - 1)) % S));
      }
    }
    cp_async_wait<0>();
    fence_proxy_async();
    for (int it = nkb > S - 1 ? nkb - (S - 1) : 0; it < nkb; ++it) mbar_arrive(bar_full + 8 * (it % S));

    }
    // epilogue: row = output channel co, columns = packed K columns of this n-tile
    mbar_wait(bar_accum, 0);
    tc_fence_after();
    const int co = (warp & 3) * 32 + lane;          // warps w and w + 4 share a TMEM lane quarter and split the 128 columns
    const uint32_t t_row = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int c_lo = mma_warp == 8 ? (warp >> 2) * 64 : 0, c_hi = mma_warp == 8 ? c_lo + 64 : 128;
    const int kcol0 = blockIdx.x * 128;
#pragma unroll 1
    for (int c0 = c_lo; c0 < c_hi; c0 += 16) {
      float v[16];
      tmem_ld16(t_row + c0, v);
      if (co < p.Cout && kcol0 + c0 < p.K_pad) {     // K_pad % 64 == 0: a 16-column group is inside or outside as a whole
        // this split's private slice, float4-COLUMN layout [K_pad / 4][Cout][4]: the warp's 32 consecutive output channels write 512
        // contiguous bytes per store (row-major [Cout][K_pad] made every store touch 32 lines, the LSU-bound pattern of the split-K slices)
        float4* o = reinterpret_cast<float4*>(p.dwp) + (size_t)blockIdx.y * p.Cout * (p.K_pad / 4) + (size_t)((kcol0 + c0) / 4) * p.Cout + co;
        o[0] = make_float4(v[0], v[1], v[2], v[3]);
        o[p.Cout] = make_float4(v[4], v[5], v[6], v[7]);
        o[2 * p.Cout] = make_float4(v[8], v[9], v[10], v[11]);
        o[3 * p.Cout] = make_float4(v[12], v[13], v[14], v[15]);
      }
    }
  } else {
    constexpr uint32_t idesc = make_idesc_bf16(128, 128, 1, 1);
    for (int it = 0; it < nkb; ++it) {
      const int s = it % S;
      const uint32_t ph = (uint32_t)((it / S) & 1);
      mbar_wait(bar_full + 8 * s, ph);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t st = tile_base + s * kWStage;
        // 16 pixels (K) per MMA = 16 rows x 128 B; MN atoms (64 channels) are kWTile apart (LBO), 8-row K groups 1024 B (SBO)
        const uint32_t alo = desc_lo(st, kWTile), blo = desc_lo(st + 2 * kWTile, kWTile), dhi = desc_hi(1024);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16_lh(tmem, alo + 128 * k, dhi, blo + 128 * k, dhi, idesc, (uint32_t)((it | k) != 0));
        umma_commit(bar_empty + 8 * s);
        if (it == nkb - 1) umma_commit(bar_accum);
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == mma_warp) tmem_dealloc<128>(tmem);
}


// ======================================================================================================= halo-resident wgrad
// EXPERIMENTAL (CisWgrad.tma == 2; written after round 1's GPU budget was spent: compiled, never run -- DESIGN.md section 6, E4).
// Swapped roles: D[kcol][co] = sum_pix x[pix + tap][c] * g[pix][co].  Per 8x8 pixel tile the CTA fetches ONE activation halo
// ((8+ex) x (8+ey) pixels x 64 channels, TMA, SWIZZLE_128B) and ONE gradient tile (8x8 pixels x 64 channels) and reads every tap
// in place: A = MN-major operand whose two 64-channel atoms are the taps 2q and 2q+1 (descriptor start = origin of tap 2q shifted
// by two tile rows per K step, LBO = distance between the two tap origins, SBO = Wh*128 between the 8-pixel rows), B = the gradient
// tile (N = Nh output channels), accumulator columns [q*Nh, (q+1)*Nh).  Relies on the tensor core applying the 128B swizzle on
// absolute address bits for MN-major operands too (tools/umma_probe_mn.cu checks exactly these descriptor forms).
// grid = (64-channel chunks of the input, pixel-tile splits, 64-channel halves of Cout); dwp layout = the tma == 1 layout.
static constexpr int kWHMaxStages = 6;
struct WgradHaloMaps {
  CUtensorMap g;                 // (C8, OW, OH, N) gradient slice, box (64, 8, 8, 1)
  CUtensorMap x[CIS_MAX_SRC];    // (C8, W, H, N) activation slices, box (64, Wh, Hh, 1)
};

__global__ void __launch_bounds__(kThreads) conv_wgrad_halo_kernel(const __grid_constant__ CisWgrad p, const __grid_constant__ WgradHaloMaps maps,
                                                                    const int Wh, const int Hh, const int hoy, const int hox,
                                                                    const int stage_bytes, const int S, const int Nh, const int ncols) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bars[2 * kWHMaxStages + 1];
  __shared__ uint32_t tmem_slot;
  __shared__ int s_off[CIS_MAX_TAPS + 1];   // tap origin inside the halo, in pixel rows of 128 B
  const uint32_t tile_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = smem_u32(&bars[0]);
  const uint32_t bar_empty = smem_u32(&bars[kWHMaxStages]);
  const uint32_t bar_accum = smem_u32(&bars[2 * kWHMaxStages]);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  pdl_launch_dependents();
  if (tid < p.ntaps) s_off[tid] = (p.dh[tid] - hoy) * Wh + (p.dw[tid] - hox);
  if (tid == p.ntaps) s_off[tid] = 0;       // partner of an unpaired last tap (its accumulator rows are never stored)
  const int halo_bytes = stage_bytes - 8192;                 // [halo (1024-rounded)] [gradient tile 8 KB]
  const int tiles_x = (p.OW + 7) / 8, tiles_y = (p.OH + 7) / 8;
  const int nkb_total = p.N * tiles_x * tiles_y;
  const int per = (nkb_total + (int)gridDim.y - 1) / (int)gridDim.y;
  const int kb0 = blockIdx.y * per;
  const int nkb = min(per, nkb_total - kb0);
  if (nkb <= 0) return;   // uniform per CTA: before any barrier / TMEM allocation
  int m_chunks = 0;
  for (int i = 0; i < p.nsrc; ++i) m_chunks += p.src[i].chunks;
  const int nch64 = (m_chunks + 7) / 8;
  const int c64 = blockIdx.x, half = blockIdx.z;
  const int npair = (p.ntaps + 1) / 2;

  if (warp == 4) {
    if (lane == 0) {
      for (int s = 0; s < S; ++s) {
        mbar_init(bar_full + 8 * s, 1);
        mbar_init(bar_empty + 8 * s, 1);
      }
      mbar_init(bar_accum, 1);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc_dyn(smem_u32(&tmem_slot), (uint32_t)ncols);
  }
  pdl_wait();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;

  if (warp < 4) {
    if (tid == 0) {
      // which concat source holds this 64-channel chunk (sources except the last are 64-channel aligned)
      int c = c64 * 8, si = 0;
      while (si < p.nsrc - 1 && c >= p.src[si].chunks) {
        c -= p.src[si].chunks;
        ++si;
      }
      int nm = p.src[0].n_mod;
      if (si == 1) nm = p.src[1].n_mod;
      if (si == 2) nm = p.src[2].n_mod;
      if (si == 3) nm = p.src[3].n_mod;
      const int tpi = tiles_x * tiles_y;
      for (int it = 0; it < nkb; ++it) {
        const int s = it % S;
        mbar_wait(bar_empty + 8 * s, (uint32_t)(((it / S) & 1) ^ 1));
        const int kb = kb0 + it;
        const int n = kb / tpi, r = kb - n * tpi;
        const int ty = r / tiles_x, tx = r - ty * tiles_x;
        const uint32_t st = tile_base + s * stage_bytes, bar = bar_full + 8 * s;
        mbar_expect_tx(bar, (uint32_t)(Wh * Hh * 128 + 8192));
        tma_load_4d(st, &maps.x[si], bar, c * 8, tx * 8 + hox, ty * 8 + hoy, nm ? (n % nm) : n);     // out-of-image pixels / channels: zeros
        tma_load_4d(st + halo_bytes, &maps.g, bar, half * 64, tx * 8, ty * 8, n);
      }
    }
    __syncwarp();
    // ---- epilogue: accumulator row r = (tap parity r / 64, input channel r % 64) of every tap pair; columns = output channels
    mbar_wait(bar_accum, 0);
    tc_fence_after();
    const int r = warp * 32 + lane;
    const int cch = r & 63;
    const uint32_t t_row = tmem + ((uint32_t)(warp * 32) << 16);
    for (int q = 0; q < npair; ++q) {
      const int t = 2 * q + (r >> 6);
      const bool tv = t < p.ntaps;
      const size_t kcol = ((size_t)t * nch64 + c64) * 64 + cch;
#pragma unroll 1
      for (int c0 = 0; c0 < Nh; c0 += 16) {
        float v[16];
        tmem_ld16(t_row + q * Nh + c0, v);     // whole-warp collective: no early exit before it
        if (!tv) continue;
        for (int e = 0; e < 16; ++e) {
          const int co = half * 64 + c0 + e;
          if (co < p.Cout) p.dwp[((size_t)blockIdx.y * p.Cout + co) * p.K_pad + kcol] = v[e];   // private slice; lanes = consecutive kcol: coalesced
        }
      }
    }
  } else {
    const uint32_t idesc = make_idesc_bf16(128, Nh, 1, 1);
    const uint32_t ahi = desc_hi((uint32_t)(Wh * 128)), bhi = desc_hi(1024);
    for (int it = 0; it < nkb; ++it) {
      const int s = it % S;
      mbar_wait(bar_full + 8 * s, (uint32_t)((it / S) & 1));
      tc_fence_after();
      if (elect_one()) {
        const uint32_t st = tile_base + s * stage_bytes;
        const uint32_t blo0 = desc_lo(st + halo_bytes, 8192);
        for (int q = 0; q < npair; ++q) {
          const int o0 = s_off[2 * q], o1 = s_off[2 * q + 1];
          const uint32_t lbo = (uint32_t)((o1 > o0 ? o1 - o0 : 1) * 128);      // distance between the two tap origins
          const uint32_t alo0 = desc_lo(st + (uint32_t)(o0 * 128), lbo);
          const uint32_t kstep = (uint32_t)(2 * Wh * 128) >> 4;                // 16 pixels = two tile rows of the halo
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_lh(tmem + q * Nh, alo0 + k * kstep, ahi, blo0 + 128 * k, bhi, idesc, (uint32_t)((it | k) != 0));
        }
        umma_commit(bar_empty + 8 * s);
        if (it == nkb - 1) umma_commit(bar_accum);
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc_dyn(tmem, (uint32_t)ncols);
}

}  // namespace cis

using namespace cis;

// Launch with programmatic stream serialization so the kernel's prologue can overlap the previous kernel's tail (the kernels call
// griddepcontrol.wait before touching dependent memory).  CIS_PDL=0 disables it.
static bool pdl_enabled() {
  static const bool on = !(getenv("CIS_PDL") && atoi(getenv("CIS_PDL")) == 0);
  return on;
}
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// launch_pdl + a thread-block cluster along grid.z (the split-K CTAs of one tile)
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl_zcluster(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cz, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = cz;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

template <int BN>
static cudaError_t launch_splitk_finish(const CisConv* d, dim3 main_grid, cudaStream_t st) {
  constexpr int G = BN / 16;
  constexpr int kBlock = (128 * G < 256) ? 128 * G : 256;
  constexpr int kSub = 128 * G / kBlock;
  const int mt = d->halo ? d->MT : 1;
  return launch_pdl(splitk_finish_kernel<BN>, dim3(main_grid.x, main_grid.y, mt * kSub), dim3(kBlock), 0, st, *d);
}

template <int BN>
static int launch_fwd(const CisConv* d, cudaStream_t st) {
  using Cfg = FwdCfg<BN>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_igemm_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem);
    if (e != cudaSuccess) return cis_set_cuda_error(e, "cudaFuncSetAttribute(conv_igemm)");
    attr_set = true;
  }
  const int M = d->N * d->OH * d->OW;
  int splits = d->splits > 1 ? d->splits : 1;
  if (splits > 1) {
    const int nkb = d->K_pad / kBK, per = (nkb + splits - 1) / splits;
    if ((!d->sk_scratch && !d->sk_cluster) || d->sk_counters || (splits - 1) * per >= nkb || (d->sk_cluster && splits > 8))
      return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm: bad split-K setup");
  }
  dim3 grid((M + kBM - 1) / kBM, d->n_tiles, splits);
  cudaError_t le = (splits > 1 && d->sk_cluster)
                       ? launch_pdl_zcluster(conv_igemm_kernel<BN>, grid, dim3(kGThreads), Cfg::kSmem, st, splits, *d)
                       : launch_pdl(conv_igemm_kernel<BN>, grid, dim3(kGThreads), Cfg::kSmem, st, *d);
  if (le != cudaSuccess) return cis_set_cuda_error(le, "launch(conv_igemm)");
  if (splits > 1 && !d->sk_cluster) {
    le = launch_splitk_finish<BN>(d, grid, st);
    if (le != cudaSuccess) return cis_set_cuda_error(le, "launch(splitk_finish)");
  }
  return cis_check_launch("conv_igemm");
}


typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}
// (C, W, H, N) bf16 map of one concat source slice; box (64, bw, bh, 1), 128B swizzle, zero OOB fill.  step = 2 selects the
// space-to-depth phase (py, px) of the image: pixel (y, x) of the map is input pixel (2y + py, 2x + px).
// step/py/px: a stride-2 phase view (coarser grid through the global strides, phase offset in the base address).
// estride: dilated layers -- ONE map per source, every estride-th pixel of a box that starts at any (phase-carrying) coordinate.
// thin: compact thin halo -- box (8, bw, bh, 1) without swizzle, one 16-byte-per-pixel plane per load (CisConv.thin).
static bool encode_src_map(CUtensorMap* m, const CisSrc& s, int N, int H, int W, int bw, int bh, int step = 1, int py = 0, int px = 0,
                           int estride = 1, bool thin = false) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) return false;
  const int nb = s.n_mod > 0 ? s.n_mod : N;
  const int Hq = (H - py + step - 1) / step, Wq = (W - px + step - 1) / step;
  if (Hq < 1 || Wq < 1) return false;
  cuuint64_t dims[4] = {(cuuint64_t)s.chunks * 8, (cuuint64_t)Wq, (cuuint64_t)Hq, (cuuint64_t)nb};
  cuuint64_t strides[3] = {(cuuint64_t)step * s.pitch * 2, (cuuint64_t)step * W * s.pitch * 2, (cuuint64_t)H * W * s.pitch * 2};
  cuuint32_t box[4] = {thin ? 8u : 64u, (cuuint32_t)(bw * estride), (cuuint32_t)(bh * estride), 1};   // extent in the un-strided pixel space
  cuuint32_t es[4] = {1, (cuuint32_t)estride, (cuuint32_t)estride, 1};
  void* base = (void*)((const char*)s.ptr + ((size_t)(py * W + px) * s.pitch + (size_t)s.c_off) * 2);
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
             thin ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B,
             CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

#ifdef CIS_TRACE
extern "C" int cis_trace_set(unsigned long long* buf, int cap) {
  cudaError_t e = cudaMemcpyToSymbol(cis::g_trace, &buf, sizeof(buf));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(cis::g_trace_cap, &cap, sizeof(cap));
  return e == cudaSuccess ? CIS_OK : cis_set_cuda_error(e, "cis_trace_set");
}
#endif

static int g_persist_mode = -1;   // -1: environment / default (1 = thin layers)
extern "C" int cis_set_persist_mode(int mode) {
  g_persist_mode = mode;
  return CIS_OK;
}

template <int BN>
static int launch_halo(const CisConv* d, cudaStream_t st) {
  const int Wh = 8 + d->ex, Hh = 16 * d->MT + d->ey, HP = Wh * Hh;
  int chunks = 0;
  for (int i = 0; i < d->nsrc; ++i) chunks += d->src[i].chunks;
  const bool thin = d->thin != 0;
  if (thin && (chunks > 2 || d->dil != 1 || d->splits > 1))
    return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm(halo): the compact thin halo takes <= 16 channels, no dilation, no split-K");
  const int halo_stage = thin ? (int)((chunks * thin_plane_bytes(HP) + 1023) & ~1023u) : (HP * 128 + 1023) & ~1023;
  const int nchunks = (chunks + 7) / 8;
  const int nsub = d->nsub > 1 ? d->nsub : 1;                  // grouped launch: grid.z = sub-problem, no split-K
  const int nsp = (nsub == 1 && d->splits > 1) ? d->splits : 1;
  const int cper = (nchunks + nsp - 1) / nsp;                  // 64-channel chunks per CTA
  const int nhs = cper * (d->nph > 1 ? d->nph : 1) > 1 ? 2 : 1; // halo stages: double-buffer only when there is a next chunk / phase to prefetch
  const int dd = d->dil;
  int tiles = 0, ntaps_max = d->ntaps;
  if (nsub > 1) {
    if (nsub > 4 || dd != 1 || d->splits > 1 || d->nph > 1) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm(halo): bad grouped launch");
    ntaps_max = 0;
    int tsum = 0;
    for (int i = 0; i < nsub; ++i) {
      const int t = ((d->sub[i].OW + 7) / 8) * ((d->sub[i].OH + 16 * d->MT - 1) / (16 * d->MT));
      if (t > tiles) tiles = t;
      if (d->sub[i].ntaps > ntaps_max) ntaps_max = d->sub[i].ntaps;
      if (d->sub[i].ntaps < 1 || d->sub[i].tap0 != tsum || !d->sub[i].wpack) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm(halo): bad sub-problem");
      tsum += d->sub[i].ntaps;
    }
    if (tsum != d->ntaps) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm(halo): sub-problem taps must add up to ntaps");
  } else {
    const int Hp0 = (d->OH + dd - 1) / dd, Wp0 = (d->OW + dd - 1) / dd;
    tiles = ((Wp0 + 7) / 8) * ((Hp0 + 16 * d->MT - 1) / (16 * d->MT));
  }
  const long ncta_all = (long)tiles * dd * dd * d->N * d->n_tiles * nsp * nsub;
  // ---- weight pipeline: G taps per stage (one bulk copy, one wait / commit of the MMA thread), BS stages
  static const int g_env = getenv("CIS_HALO_G") ? atoi(getenv("CIS_HALO_G")) : 0;            // experiments: force the group size
  static const int stage_kb = getenv("CIS_HALO_STAGE_KB") ? atoi(getenv("CIS_HALO_STAGE_KB")) : 48;
  const int kB = thin ? BN * 32 : BN * 128;     // weight bytes per tap (compact: per K=16 MMA)
  int G = g_env > 0 ? g_env : (stage_kb * 1024) / kB;
  if (G < 1) G = 1;
  if (G > ntaps_max) G = ntaps_max;
  const int fixed = nhs * halo_stage + HP * 4 + 1024;
  // two co-resident CTAs per SM overlap one CTA's epilogue with the other's main loop -- when the grid has that many CTAs
  static const int lim_small_kb = getenv("CIS_HALO_SMALL_KB") ? atoi(getenv("CIS_HALO_SMALL_KB")) : 226;   // grids of <= 148 CTAs
  static const int lim_kb_wide = getenv("CIS_HALO_LIMIT_KB") ? atoi(getenv("CIS_HALO_LIMIT_KB")) : 113;
  static const int lim_kb_thin = getenv("CIS_HALO_LIMIT_THIN_KB") ? atoi(getenv("CIS_HALO_LIMIT_THIN_KB")) : 113;   // BN <= 32
  const int lim_kb = BN <= 32 ? lim_kb_thin : lim_kb_wide;
  int limit = (ncta_all > 148 && fixed + 2 * kB <= lim_kb * 1024) ? lim_kb * 1024 : 226 * 1024;
  if (ncta_all <= 148 && fixed + 2 * kB <= lim_small_kb * 1024) limit = lim_small_kb * 1024;
  while (G > 1 && fixed + 2 * G * kB > limit) --G;
  const int groups = cper * ((nsub > 1 ? 1 : (ntaps_max + G - 1) / G));   // pipeline stages one CTA walks (grouped: at least one per chunk)
  int BS = (limit - fixed) / (G * kB);
  if (BS > (ncta_all > 148 ? 4 : kHaloMaxBStages)) BS = ncta_all > 148 ? 4 : kHaloMaxBStages;
  if (BS > groups) BS = groups;
  if (BS < 1) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_conv_igemm(halo): tile does not fit shared memory");
  int smem = fixed + BS * G * kB;
  if (nsp > 1 && d->sk_cluster && smem < d->MT * kBM * BN * 4 + 1024) smem = d->MT * kBM * BN * 4 + 1024;   // fp32 staging tiles of the cluster reduction
  if (smem > 226 * 1024) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_conv_igemm(halo): cluster split-K staging does not fit shared memory");
  static int attr_smem = 0;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(conv_halo_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return cis_set_cuda_error(e, "cudaFuncSetAttribute(conv_halo)");
    attr_smem = smem;
  }

  int splits = d->splits > 1 ? d->splits : 1;
  if (splits > 1) {
    const int per = (nchunks + splits - 1) / splits;
    if ((!d->sk_scratch && !d->sk_cluster) || d->sk_counters || (splits - 1) * per >= nchunks || (d->sk_cluster && splits > 8))
      return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm(halo): bad split-K setup");
  }
  dim3 grid(tiles * dd * dd * d->N, d->n_tiles, nsub > 1 ? nsub : splits);
  // TMA halo path: undilated, every concat source except the last a multiple of 64 channels (a chunk never straddles sources)
  HaloMaps maps;
  const int nph = d->nph > 1 ? d->nph : 1;
  static const int dil_tma = getenv("CIS_DIL_TMA") ? atoi(getenv("CIS_DIL_TMA")) : 1;
  int use_tma = ((d->dil == 1 || dil_tma) && Wh * d->dil <= 256 && Hh * d->dil <= 256) ? 1 : 0;
  for (int i = 0; use_tma && !thin && i < d->nsrc - 1; ++i)     // (compact planes are 8 channels: they never straddle sources)
    if (d->src[i].chunks % 8) use_tma = 0;
  for (int i = 0; use_tma && i < d->nsrc; ++i) {
    if (((uintptr_t)d->src[i].ptr + (size_t)d->src[i].c_off * 2) % 16) use_tma = 0;
    for (int ph = 0; use_tma && ph < nph; ++ph)
      if (!encode_src_map(&maps.m[i * nph + ph], d->src[i], d->N, d->H, d->W, Wh, Hh, nph > 1 ? 2 : 1, ph >> 1, ph & 1, d->dil, thin)) use_tma = 0;
  }
  if (!use_tma) memset(&maps, 0, sizeof(maps));
  if (thin && !use_tma) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_conv_igemm(halo): the compact thin halo needs the TMA halo path");
  if (nph > 1 && !use_tma) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_conv_igemm(halo): stride-2 phases need the TMA halo path");
  // persistent variant (conv_halo_persist_kernel): layers with many tiles per SM.  CIS_PERSIST_MODE / cis_set_persist_mode:
  //   0 off | 1 (default) layers whose whole weight set stays resident in shared memory and that have >= 2 tiles per SM |
  //   2 every eligible layer (tests) | 3 every layer whose weight set fits, whatever the tile count (tests)
  const int persist_mode = g_persist_mode >= 0 ? g_persist_mode : (getenv("CIS_PERSIST_MODE") ? atoi(getenv("CIS_PERSIST_MODE")) : 1);
  static const int p_min_tiles = getenv("CIS_PERSIST_MIN_TILES") ? atoi(getenv("CIS_PERSIST_MIN_TILES")) : 296;
  static const int p_ws_kb = getenv("CIS_PERSIST_WS_KB") ? atoi(getenv("CIS_PERSIST_WS_KB")) : 112;
  if (persist_mode > 0 && use_tma && d->n_tiles == 1 && splits == 1 && nph == 1 && nsub == 1 && dd == 1) {
    const int total = tiles * d->N;
    const int per_tile = nchunks * d->ntaps;
    const int AS = (2 * d->MT * BN <= 512) ? 2 : 1;
    const int ws_bytes = per_tile * kB;
    int p_nhs = nchunks >= 3 ? 4 : 3;
    while (p_nhs > 2 && p_nhs * halo_stage + 1024 + (ws_bytes <= p_ws_kb * 1024 ? ws_bytes : 2 * G * kB) > 226 * 1024) --p_nhs;
    const bool ws_fits = ws_bytes <= p_ws_kb * 1024 && p_nhs * halo_stage + 1024 + ws_bytes <= 226 * 1024;
    const bool take = persist_mode == 2 || (persist_mode == 3 && ws_fits) || (persist_mode == 1 && ws_fits && total >= p_min_tiles);
    int p_bs = 0, p_smem = 0;
    if (ws_fits) {
      p_bs = 1;
      p_smem = p_nhs * halo_stage + 1024 + ws_bytes;
    } else {
      p_bs = (226 * 1024 - p_nhs * halo_stage - 1024) / (G * kB);
      if (p_bs > 4) p_bs = 4;
      p_smem = p_nhs * halo_stage + 1024 + p_bs * G * kB;
    }
    if (take && p_bs >= (ws_fits ? 1 : 2)) {
      static int attr_p = 0;   // largest dynamic-smem limit set so far on conv_halo_persist_kernel<BN>
      if (p_smem > attr_p) {
        cudaError_t e = cudaFuncSetAttribute(conv_halo_persist_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, p_smem);
        if (e != cudaSuccess) return cis_set_cuda_error(e, "cudaFuncSetAttribute(conv_halo_persist)");
        attr_p = p_smem;
      }
      const int want = AS * d->MT * BN;
      const int tcols = want <= 32 ? 32 : want <= 64 ? 64 : want <= 128 ? 128 : want <= 256 ? 256 : 512;
      int cps = (227 * 1024) / (p_smem + 1024);          // co-resident persistent CTAs per SM: shared memory, TMEM columns, threads
      if (cps > 512 / tcols) cps = 512 / tcols;
      if (cps > 2048 / kPThreads) cps = 2048 / kPThreads;
      if (cps > 2) cps = 2;
      if (cps < 1) cps = 1;
      int g = total < 148 * cps ? total : 148 * cps;
      cudaError_t le = launch_pdl(conv_halo_persist_kernel<BN>, dim3(g), dim3(kPThreads), p_smem, st, *d, halo_stage, p_bs, p_nhs, AS, G, maps,
                                  ws_fits ? 1 : 0);
      if (le != cudaSuccess) return cis_set_cuda_error(le, "launch(conv_halo_persist)");
      return cis_check_launch("conv_halo_persist");
    }
  }
  cudaError_t le = (splits > 1 && d->sk_cluster)
                       ? launch_pdl_zcluster(conv_halo_kernel<BN>, grid, dim3(HaloCfg<BN>::kThreads), smem, st, splits, *d, halo_stage, BS, nhs, maps, use_tma, G)
                       : launch_pdl(conv_halo_kernel<BN>, grid, dim3(HaloCfg<BN>::kThreads), smem, st, *d, halo_stage, BS, nhs, maps, use_tma, G);
  if (le != cudaSuccess) return cis_set_cuda_error(le, "launch(conv_halo)");
  if (splits > 1 && !d->sk_cluster) {
    le = launch_splitk_finish<BN>(d, grid, st);
    if (le != cudaSuccess) return cis_set_cuda_error(le, "launch(splitk_finish)");
  }
  return cis_check_launch("conv_halo");
}

extern "C" int cis_conv_igemm(const CisConv* d, cis_stream_t stream) {
  if (!d || d->ntaps < 1 || d->ntaps > CIS_MAX_TAPS || d->nsrc < 1 || d->nsrc > CIS_MAX_SRC || d->K_pad % 64 != 0 || d->K_pad <= 0 ||
      d->n_tiles < 1 || !d->wpack)
    return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm: bad descriptor");
  int chunks = 0;
  for (int i = 0; i < d->nsrc; ++i) {
    if ((d->src[i].pitch | d->src[i].c_off) & 7) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm: source pitch/c_off must be multiples of 8");
    chunks += d->src[i].chunks;
  }
  if (d->ntaps * chunks * 8 > d->K_pad) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm: K_pad smaller than taps*channels");
  if (d->mode == 1 && !d->outf) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm: mode 1 needs outf");
  if ((d->add_pre || d->add_post) && (((d->add_pre_pitch | d->add_pre_coff | d->add_post_pitch | d->add_post_coff | d->out_ch) & 7) != 0))
    return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm: residual slices must be 8-channel aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (d->halo) {
    if (d->MT < 1 || d->MT > 4 || d->MT * d->BN > 512 || d->dil < 1 || d->sh != 1 || d->sw != 1 || d->ey < 0 || d->ex < 0 ||
        (d->dil > 1 && (d->OH != d->H || d->OW != d->W)) || (d->nph > 1 && (d->nph != 4 || d->dil != 1 || d->ph_tap[0] != 0 || d->ph_tap[4] != d->ntaps)))
      return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_igemm(halo): bad tile parameters");
    switch (d->BN) {
      case 16: return launch_halo<16>(d, st);
      case 32: return launch_halo<32>(d, st);
      case 64: return launch_halo<64>(d, st);
      case 128: return launch_halo<128>(d, st);
      default: return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_conv_igemm: BN must be 16/32/64/128");
    }
  }
  switch (d->BN) {
    case 16: return launch_fwd<16>(d, st);
    case 32: return launch_fwd<32>(d, st);
    case 64: return launch_fwd<64>(d, st);
    case 128: return launch_fwd<128>(d, st);
    default: return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_conv_igemm: BN must be 16/32/64/128");
  }
}

// Halo-resident swapped wgrad (CisWgrad.tma == 2, experimental).  Eligibility is re-checked here; the engine falls back to tma = 1.
static int launch_wgrad_halo(const CisWgrad* d, cudaStream_t st) {
  if (d->sh != 1 || d->sw != 1) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_wgrad(halo): needs a stride-1 layer");
  int chunks = 0;
  for (int i = 0; i < d->nsrc; ++i) chunks += d->src[i].chunks;
  for (int i = 0; i < d->nsrc - 1; ++i)
    if (d->src[i].chunks % 8) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_wgrad(halo): needs 64-channel aligned concat sources");
  const int nch64 = (chunks + 7) / 8;
  int hoy = d->dh[0], hox = d->dw[0], my = d->dh[0], mx = d->dw[0];
  for (int t = 1; t < d->ntaps; ++t) {
    if (d->dh[t] < hoy) hoy = d->dh[t];
    if (d->dw[t] < hox) hox = d->dw[t];
    if (d->dh[t] > my) my = d->dh[t];
    if (d->dw[t] > mx) mx = d->dw[t];
  }
  for (int t = 1; t < d->ntaps; ++t)    // pairs (2q, 2q+1) need increasing origins: taps are listed row-major
    if ((d->dh[t] - hoy) * 1024 + (d->dw[t] - hox) <= (d->dh[t - 1] - hoy) * 1024 + (d->dw[t - 1] - hox))
      return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_wgrad(halo): taps must be listed in increasing row-major order");
  const int Wh = 8 + (mx - hox), Hh = 8 + (my - hoy);
  if (Wh > 256 || Hh > 256) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_conv_wgrad(halo): tap extent too large");
  const int halo_bytes = (Wh * Hh * 128 + 1023) & ~1023;
  const int stage = halo_bytes + 8192;
  const int nhalf = d->Cout > 64 ? 2 : 1;
  int Nh = d->Cout > 64 ? 64 : ((d->Cout + 15) & ~15);
  const int npair = (d->ntaps + 1) / 2;
  const int want = npair * Nh;
  if (want > 512) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_conv_wgrad(halo): accumulators exceed TMEM");
  const int ncols = want <= 32 ? 32 : want <= 64 ? 64 : want <= 128 ? 128 : want <= 256 ? 256 : 512;
  int S = (200 * 1024) / stage;
  if (S > kWHMaxStages) S = kWHMaxStages;
  if (S > 4 && ncols <= 256) S = 4;       // leave room for a second co-resident CTA when TMEM allows one
  if (S < 2) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_conv_wgrad(halo): halo does not fit shared memory");
  const int smem = S * stage + 1024;
  static int attr_smem = 0;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return cis_set_cuda_error(e, "cudaFuncSetAttribute(conv_wgrad_halo)");
    attr_smem = smem;
  }
  if (d->K_pad < d->ntaps * nch64 * 64) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_wgrad(halo): K_pad smaller than taps * 64-channel groups");
  WgradHaloMaps maps;
  memset(&maps, 0, sizeof(maps));
  CisSrc gs;
  gs.ptr = d->g; gs.pitch = d->g_pitch; gs.c_off = d->g_coff; gs.chunks = d->g_chunks; gs.n_mod = 0;
  bool ok = encode_src_map(&maps.g, gs, d->N, d->OH, d->OW, 8, 8);
  for (int i = 0; ok && i < d->nsrc; ++i) ok = encode_src_map(&maps.x[i], d->src[i], d->N, d->H, d->W, Wh, Hh);
  if (!ok) return cis_set_error(CIS_ERR_CUDA, "cis_conv_wgrad(halo): cuTensorMapEncodeTiled failed / unavailable");
  dim3 grid(nch64, d->splits, nhalf);
  cudaError_t le = launch_pdl(conv_wgrad_halo_kernel, grid, dim3(kThreads), (size_t)smem, st, *d, maps, Wh, Hh, hoy, hox, stage, S, Nh, ncols);
  if (le != cudaSuccess) return cis_set_cuda_error(le, "launch(conv_wgrad_halo)");
  return cis_check_launch("conv_wgrad_halo");
}

extern "C" int cis_conv_wgrad(const CisWgrad* d, cis_stream_t stream) {
  if (!d || d->ntaps < 1 || d->ntaps > CIS_MAX_TAPS || d->nsrc < 1 || d->nsrc > CIS_MAX_SRC || d->K_pad % 64 != 0 || d->Cout < 1 ||
      d->Cout > 128 || d->splits < 1 || !d->g || !d->dwp)
    return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_wgrad: bad descriptor");
  {
    // every split must own at least one reduction block: its private slice of dwp is only defined if the CTA runs
    const long M = (long)d->N * d->OH * d->OW;
    const long nkb_total = d->tma ? (long)d->N * ((d->OW + 7) / 8) * ((d->OH + 7) / 8) : (M + 63) / 64;
    const long per = (nkb_total + d->splits - 1) / d->splits;
    if ((long)(d->splits - 1) * per >= nkb_total) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_wgrad: a split would own no reduction block");
  }
  if (d->tma == 2) return launch_wgrad_halo(d, (cudaStream_t)stream);
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWSmem);
    if (e != cudaSuccess) return cis_set_cuda_error(e, "cudaFuncSetAttribute(conv_wgrad)");
    attr_set = true;
  }
  WgradMaps maps;
  memset(&maps, 0, sizeof(maps));
  if (d->tma) {
    if (d->sh != 1 || d->sw != 1) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_wgrad: TMA path needs a stride-1 layer");
    for (int i = 0; i < d->nsrc - 1; ++i)
      if (d->src[i].chunks % 8) return cis_set_error(CIS_ERR_BAD_ARG, "cis_conv_wgrad: TMA path needs 64-channel aligned concat sources");
    CisSrc gs;
    gs.ptr = d->g; gs.pitch = d->g_pitch; gs.c_off = d->g_coff; gs.chunks = d->g_chunks; gs.n_mod = 0;
    bool ok = encode_src_map(&maps.g, gs, d->N, d->OH, d->OW, 8, 8);
    for (int i = 0; ok && i < d->nsrc; ++i) ok = encode_src_map(&maps.x[i], d->src[i], d->N, d->H, d->W, 8, 8);
    if (!ok) return cis_set_error(CIS_ERR_CUDA, "cis_conv_wgrad: cuTensorMapEncodeTiled failed / unavailable");
  }
  dim3 grid((d->K_pad + 127) / 128, d->splits);
  cudaError_t le = launch_pdl(conv_wgrad_kernel, grid, dim3(d->tma ? kThreads : kGThreads), kWSmem, (cudaStream_t)stream, *d, maps);
  if (le != cudaSuccess) return cis_set_cuda_error(le, "launch(conv_wgrad)");
  return cis_check_launch("conv_wgrad");
}
