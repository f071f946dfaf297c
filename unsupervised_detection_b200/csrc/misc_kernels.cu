// HBM-bound kernels of the hot path: parameter packing, activation-gradient helpers, TF-1.13 resampling ops, the fused
// PWC-Net warp + cost volume, the fused mask (x) flow + Charbonnier loss, and clip + TF-Adam.
// Reference call sites are cited per kernel; semantics follow SURVEY.md Appendix A.
#include "ptx.cuh"
#include "../../include/cis_b200.h"
#include "common.cuh"
#include <math.h>

namespace cis {

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  f[0] = bf16lo(u.x); f[1] = bf16hi(u.x); f[2] = bf16lo(u.y); f[3] = bf16hi(u.y);
  f[4] = bf16lo(u.z); f[5] = bf16hi(u.z); f[6] = bf16lo(u.w); f[7] = bf16hi(u.w);
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  return make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------ weights
// The five parameter-space ops (BN fold, two weight packs, gradient un-pack, BN chain rule) exist as single launches AND as one
// multi-job launch (cis_param_multi): blockIdx.y selects a job from a device-side table, so the ~75 per-layer launches that follow
// every optimiser step and the ~35 that end every backward pass become a handful.
__device__ __forceinline__ void pack_weights_body(size_t i, const float* __restrict__ w, const int* __restrict__ kmap, int K_pad, int rows, int cout,
                                                  int sn, const int* __restrict__ nmap, bf16* __restrict__ wp) {
  if (i >= (size_t)rows * K_pad) return;
  const int n = (int)(i / K_pad), k = (int)(i % K_pad);
  const int km = kmap[k];
  const int ne = nmap ? nmap[n] : (n < cout ? n : -1);
  const float v = (km >= 0 && ne >= 0) ? w[(size_t)km + (size_t)ne * sn] : 0.f;
  wp[i] = __float2bfloat16(v);
}
// Pre-swizzled weight tiles for the halo kernel: block (ny, cc, t) = BN rows x 128 B, row n holds K = 64 channels of chunk cc for
// tap t with the SWIZZLE_128B pattern already applied (16-byte chunk index ^= n & 7), so a plain bulk copy lands the UMMA layout.
// layout 1 (compact thin halo, CisConv.thin): cin8 = 16 K positions per "tap" (= one K=16 MMA), block t = BN x 32 B in the no-swizzle
// K-major canonical layout [K half][n][8]: core matrices of 8 n-rows x 16 B, 128 B apart along n (SBO), BN x 16 B apart along K (LBO).
__device__ __forceinline__ int tiled_kk(int q, int BN, int layout, int& n) {
  if (layout) {
    n = (q >> 3) % BN;
    return ((q / (BN * 8)) << 3) | (q & 7);
  }
  n = q >> 6;
  const int pos = q & 63;                    // physical element position inside the 128-byte row
  return (((pos >> 3) ^ (n & 7)) << 3) | (pos & 7);   // logical channel within the chunk
}
__device__ __forceinline__ void pack_weights_tiled_body(size_t i, const float* __restrict__ w, const int* __restrict__ kmap, int cin8, int ntaps,
                                                        int n_tiles, int BN, int cout, int sn, const int* __restrict__ nmap,
                                                        bf16* __restrict__ out, int layout) {
  const int nchunks = (cin8 + 63) / 64;
  const int KT = layout ? 16 : 64;
  const size_t total = (size_t)n_tiles * nchunks * ntaps * BN * KT;
  if (i >= total) return;
  size_t r = i / ((size_t)BN * KT);
  int n;
  const int kk = tiled_kk((int)(i % ((size_t)BN * KT)), BN, layout, n);
  const int t = (int)(r % ntaps); r /= ntaps;
  const int cc = (int)(r % nchunks);
  const int ny = (int)(r / nchunks);
  const int c = cc * 64 + kk;
  float v = 0.f;
  if (c < cin8) {
    const int km = kmap[t * cin8 + c];
    const int ng = ny * BN + n;
    const int ne = nmap ? nmap[ng] : (ng < cout ? ng : -1);
    if (km >= 0 && ne >= 0) v = w[(size_t)km + (size_t)ne * sn];
  }
  out[i] = __float2bfloat16(v);
}
// Forward orientation (sn == 1: the fp32 master weights are HWIO, output channel fastest): one block per (ny, cc, t) tile of BN x 64
// elements, read along n (contiguous in HWIO), transposed through shared memory, written along k (contiguous in the tile).  The flat
// form above reads a column of the [tap*cin][cout] matrix per warp: 4 useful bytes per 32-byte sector.  tile: >= 64 * (BN + 1) floats.
__device__ __forceinline__ void pack_weights_tiled_tile(int blk, const float* __restrict__ w, const int* __restrict__ kmap, int cin8, int ntaps,
                                                        int n_tiles, int BN, int cout, const int* __restrict__ nmap, bf16* __restrict__ out,
                                                        float* tile, int layout) {
  const int nchunks = (cin8 + 63) / 64;
  const int KT = layout ? 16 : 64;
  const int t = blk % ntaps;
  const int r = blk / ntaps;
  const int cc = r % nchunks, ny = r / nchunks;
  const int ld = BN + 1;
  for (int idx = threadIdx.x; idx < BN * KT; idx += blockDim.x) {
    const int n = idx % BN, kk = idx / BN;
    const int c = cc * 64 + kk;
    float v = 0.f;
    if (c < cin8) {
      const int km = kmap[t * cin8 + c];
      const int ng = ny * BN + n;
      const int ne = nmap ? nmap[ng] : (ng < cout ? ng : -1);
      if (km >= 0 && ne >= 0) v = w[(size_t)km + ne];
    }
    tile[kk * ld + n] = v;
  }
  __syncthreads();
  bf16* o = out + (size_t)blk * BN * KT;
  for (int idx = threadIdx.x; idx < BN * KT; idx += blockDim.x) {
    int n;
    const int kk = tiled_kk(idx, BN, layout, n);
    o[idx] = __float2bfloat16(tile[kk * ld + n]);
  }
}
__device__ __forceinline__ void unpack_wgrad_body(size_t i, const float* __restrict__ dwp, const int* __restrict__ kmap, int K_pad, int cout,
                                                  int nsplit, float* __restrict__ dw, const float* __restrict__ colpart, int nblocks, int nch,
                                                  float* __restrict__ db, int layout) {
  const size_t nw = (size_t)cout * K_pad;
  if (i < nw) {
    // slice element i -> (output channel n, packed column k): layout 0 = [cout][K_pad] (halo-resident wgrad), layout 1 = float4 columns
    // [K_pad / 4][cout][4] (gather / TMA-tile wgrad kernels)
    int n, k;
    if (layout == 0) {
      n = (int)(i / K_pad);
      k = (int)(i % K_pad);
    } else {
      const size_t g4 = i / ((size_t)cout * 4);
      const int rem = (int)(i - g4 * cout * 4);
      n = rem >> 2;
      k = (int)g4 * 4 + (rem & 3);
    }
    const int km = kmap[k];
    if (km < 0) return;
    // fixed-order sum of the private split-K slices; 8 independent loads in flight per thread
    float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const float* q = dwp + i;
    int s = 0;
    for (; s + 8 <= nsplit; s += 8) {
      float t[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) t[u] = __ldcg(q + (size_t)(s + u) * nw);
#pragma unroll
      for (int u = 0; u < 8; ++u) a[u] += t[u];
    }
    for (; s < nsplit; ++s) a[0] += __ldcg(q + (size_t)s * nw);
    dw[(size_t)km + n] = ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
  } else if (colpart != nullptr && i - nw < (size_t)nch) {
    const int c = (int)(i - nw);
    float a = 0.f;
    for (int b = 0; b < nblocks; ++b) a += __ldcg(colpart + (size_t)b * nch + c);
    db[c] = a;
  }
}
#define BN_RSQRT 0.99950037468777323f /* 1/sqrt(1 + 1e-3): tf.layers.batch_normalization defaults, convolution_utils.py:50 */
__device__ __forceinline__ void bn_fold_body(size_t i, const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ gamma,
                                             const float* __restrict__ beta, size_t nw, int cout, float* __restrict__ w_eff,
                                             float* __restrict__ b_eff) {
  if (i < nw) w_eff[i] = w[i] * gamma[i % cout] * BN_RSQRT;
  if (i < (size_t)cout) b_eff[i] = bias[i] * gamma[i] * BN_RSQRT + beta[i];
}
// one 256-thread block per 8 output channels: thread = (channel co0 + tid % 8, row lane tid / 8), so a row of 8 channels is one 32-byte
// sector and every byte fetched is used.  (r02: one block per channel walked a column of the [rows][cout] matrix -- 4 useful bytes per
// sector, 96 us for the generator's 1.45 M parameters; this form moves the same data in ~10 us.)  Fixed summation order.
static constexpr int kBnChainCo = 8;
__device__ __forceinline__ void bn_chain_body(int blk, const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ gamma,
                                              float* __restrict__ dwe, const float* __restrict__ dbe, size_t nw, int cout,
                                              float* __restrict__ dbias, float* __restrict__ dgamma, float* __restrict__ dbeta, float* red) {
  const int rows = (int)(nw / cout);
  const int cl = threadIdx.x & 7, rl = threadIdx.x >> 3;          // 8 channels x 32 row lanes
  const int co = blk * kBnChainCo + cl;
  const bool ok = co < cout;
  float acc = 0.f;
  if (ok)
    for (int r = rl; r < rows; r += 32) acc += dwe[(size_t)r * cout + co] * w[(size_t)r * cout + co];
  red[rl * 8 + cl] = acc;
  __syncthreads();
  float g = 0.f;
  if (ok) {
    g = gamma[co] * BN_RSQRT;
    if (rl == 0) {
      float v = 0.f;
      for (int q = 0; q < 32; ++q) v += red[q * 8 + cl];
      dgamma[co] = BN_RSQRT * (v + dbe[co] * bias[co]);
      dbias[co] = dbe[co] * g;
      dbeta[co] = dbe[co];
    }
    for (int r = rl; r < rows; r += 32) dwe[(size_t)r * cout + co] *= g;
  }
}
__global__ void pack_weights_kernel(const float* __restrict__ w, const int* __restrict__ kmap, int K_pad, int rows, int cout, int sn,
                                    const int* __restrict__ nmap, bf16* __restrict__ wp) {
  pdl_launch_dependents();
  pdl_wait();
  pack_weights_body((size_t)blockIdx.x * blockDim.x + threadIdx.x, w, kmap, K_pad, rows, cout, sn, nmap, wp);
}
__global__ void pack_weights_tiled_kernel(const float* __restrict__ w, const int* __restrict__ kmap, int cin8, int ntaps, int n_tiles, int BN,
                                          int cout, int sn, const int* __restrict__ nmap, bf16* __restrict__ out, int layout) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float tile[64 * 129];
  if (sn == 1) pack_weights_tiled_tile(blockIdx.x, w, kmap, cin8, ntaps, n_tiles, BN, cout, nmap, out, tile, layout);
  else pack_weights_tiled_body((size_t)blockIdx.x * blockDim.x + threadIdx.x, w, kmap, cin8, ntaps, n_tiles, BN, cout, sn, nmap, out, layout);
}
__global__ void unpack_wgrad_kernel(const float* __restrict__ dwp, const int* __restrict__ kmap, int K_pad, int cout, int nsplit,
                                    float* __restrict__ dw, const float* __restrict__ colpart, int nblocks, int nch, float* __restrict__ db,
                                    int layout) {
  pdl_launch_dependents();
  pdl_wait();
  unpack_wgrad_body((size_t)blockIdx.x * blockDim.x + threadIdx.x, dwp, kmap, K_pad, cout, nsplit, dw, colpart, nblocks, nch, db, layout);
}
__global__ void bn_fold_kernel(const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ gamma,
                               const float* __restrict__ beta, size_t nw, int cout, float* __restrict__ w_eff, float* __restrict__ b_eff) {
  pdl_launch_dependents();
  pdl_wait();
  bn_fold_body((size_t)blockIdx.x * blockDim.x + threadIdx.x, w, bias, gamma, beta, nw, cout, w_eff, b_eff);
}
__global__ void bn_chain_kernel(const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ gamma,
                                float* __restrict__ dwe, const float* __restrict__ dbe, size_t nw, int cout, float* __restrict__ dbias,
                                float* __restrict__ dgamma, float* __restrict__ dbeta) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[256];
  bn_chain_body(blockIdx.x, w, bias, gamma, dwe, dbe, nw, cout, dbias, dgamma, dbeta, red);
}
// multi-job form: a flat 1-D grid; job j owns blocks [jobs[j].i[7], jobs[j+1].i[7]) (binary search), fields in the argument order of the
// single-launch entry points
__global__ void param_multi_kernel(const CisParamJob* __restrict__ jobs, int njobs) {
  pdl_launch_dependents();
  pdl_wait();
  int lo = 0, hi = njobs - 1;
  while (lo < hi) {                       // last job whose first block is <= blockIdx.x
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].i[7] <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const CisParamJob j = jobs[lo];
  const int blk = (int)blockIdx.x - j.i[7];
  const size_t i = (size_t)blk * blockDim.x + threadIdx.x;
  __shared__ float red[256];
  __shared__ float tile[64 * 129];
  switch (j.kind) {
    case CIS_JOB_PACK:
      pack_weights_body(i, (const float*)j.p[0], (const int*)j.p[1], j.i[0], j.i[1], j.i[2], j.i[3], (const int*)j.p[2], (bf16*)j.p[3]);
      break;
    case CIS_JOB_PACK_TILED:
      if (j.i[5] == 1)       // forward orientation: one block per tile, transposed through shared memory
        pack_weights_tiled_tile(blk, (const float*)j.p[0], (const int*)j.p[1], j.i[0], j.i[1], j.i[2], j.i[3], j.i[4], (const int*)j.p[2],
                                (bf16*)j.p[3], tile, j.i[6]);
      else
        pack_weights_tiled_body(i, (const float*)j.p[0], (const int*)j.p[1], j.i[0], j.i[1], j.i[2], j.i[3], j.i[4], j.i[5], (const int*)j.p[2],
                                (bf16*)j.p[3], j.i[6]);
      break;
    case CIS_JOB_UNPACK:
      unpack_wgrad_body(i, (const float*)j.p[0], (const int*)j.p[1], j.i[0], j.i[1], j.i[2], (float*)j.p[2], (const float*)j.p[3], j.i[3], j.i[4],
                        (float*)j.p[4], j.i[5]);
      break;
    case CIS_JOB_BN_FOLD:
      bn_fold_body(i, (const float*)j.p[0], (const float*)j.p[1], (const float*)j.p[2], (const float*)j.p[3], (size_t)j.n, j.i[0], (float*)j.p[4],
                   (float*)j.p[5]);
      break;
    case CIS_JOB_BN_CHAIN:      // one block per 8 output channels; the host gives the job exactly ceil(cout / 8) blocks
      bn_chain_body(blk, (const float*)j.p[0], (const float*)j.p[1], (const float*)j.p[2], (float*)j.p[3], (const float*)j.p[4], (size_t)j.n,
                    j.i[0], (float*)j.p[5], (float*)j.p[6], (float*)j.p[7], red);
      break;
  }
}

// ------------------------------------------------------------------------------------------------ gradient helpers
__global__ void dact_mul_kernel(bf16* g, int gp, int gc, const bf16* __restrict__ y, int yp, int yc, const bf16* __restrict__ res, int rp,
                                int rc, size_t npix, int chunks, int act, float alpha) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix * chunks) return;
  const size_t pix = i / chunks;
  const int c = (int)(i % chunks) * 8;
  uint4* gpp = reinterpret_cast<uint4*>(g + pix * gp + gc + c);
  float gv[8], yv[8], rv[8];
  unpack8(*gpp, gv);
  unpack8(*reinterpret_cast<const uint4*>(y + pix * yp + yc + c), yv);
  if (res) {
    unpack8(*reinterpret_cast<const uint4*>(res + pix * rp + rc + c), rv);
#pragma unroll
    for (int e = 0; e < 8; ++e) yv[e] -= rv[e];
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float u = yv[e];
    const float d = (act == CIS_ACT_ELU) ? (u > 0.f ? 1.f : u + 1.f) : (u > 0.f ? 1.f : alpha);
    gv[e] *= d;
  }
  *gpp = pack8(gv);
}
__global__ void add_slice_kernel(bf16* dst, int dp, int dc, const bf16* __restrict__ src, int sp, int sc, size_t npix, int chunks, int reps,
                                 int accumulate) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix * chunks) return;
  const size_t pix = i / chunks;
  const int c = (int)(i % chunks) * 8;
  float a[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t[8];
  uint4* d = reinterpret_cast<uint4*>(dst + pix * dp + dc + c);
  if (accumulate) unpack8(*d, a);
  for (int j = 0; j < reps; ++j) {
    unpack8(*reinterpret_cast<const uint4*>(src + (pix + (size_t)j * npix) * sp + sc + c), t);
#pragma unroll
    for (int e = 0; e < 8; ++e) a[e] += t[e];
  }
  *d = pack8(a);
}
// part[blockIdx.x][c] = sum over this block's pixels of g[pix][c].  blockDim = 256 = P pixel lanes x chunks (chunks <= 32).
__global__ void colsum_kernel(const bf16* __restrict__ g, int gp, int gc, size_t npix, int nch, int chunks, float* __restrict__ part) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];  // [P][chunks*8]
  const int P = blockDim.x / chunks;
  const int ck = threadIdx.x % chunks, pl = threadIdx.x / chunks;
  float a[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t[8];
  if (pl < P) {
    for (size_t p = (size_t)blockIdx.x * P + pl; p < npix; p += (size_t)gridDim.x * P) {
      unpack8(*reinterpret_cast<const uint4*>(g + p * gp + gc + ck * 8), t);
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] += t[e];
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) sm[pl * chunks * 8 + ck * 8 + e] = a[e];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < nch; c += blockDim.x) {
    float s = 0.f;
    for (int q = 0; q < P; ++q) s += sm[q * chunks * 8 + c];
    part[(size_t)blockIdx.x * nch + c] = s;
  }
}

// dact_mul + colsum in one pass (layers that have an activation AND accumulate a bias gradient in this backward pass): g *= act'(y - res)
// in place, part[blockIdx.x][c] = this block's column sums of the ROUNDED product (what a separate colsum launch would read back).
__global__ void dact_colsum_kernel(bf16* g, int gp, int gc, const bf16* __restrict__ y, int yp, int yc, const bf16* __restrict__ res, int rp,
                                   int rc, size_t npix, int nch, int chunks, int act, float alpha, float* __restrict__ part) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];  // [P][chunks*8]
  const int P = blockDim.x / chunks;
  const int ck = threadIdx.x % chunks, pl = threadIdx.x / chunks;
  float a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (pl < P) {
    for (size_t p = (size_t)blockIdx.x * P + pl; p < npix; p += (size_t)gridDim.x * P) {
      uint4* gpp = reinterpret_cast<uint4*>(g + p * gp + gc + ck * 8);
      float gv[8], yv[8], rv[8];
      unpack8(*gpp, gv);
      unpack8(*reinterpret_cast<const uint4*>(y + p * yp + yc + ck * 8), yv);
      if (res) {
        unpack8(*reinterpret_cast<const uint4*>(res + p * rp + rc + ck * 8), rv);
#pragma unroll
        for (int e = 0; e < 8; ++e) yv[e] -= rv[e];
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float u = yv[e];
        gv[e] *= (act == CIS_ACT_ELU) ? (u > 0.f ? 1.f : u + 1.f) : (u > 0.f ? 1.f : alpha);
      }
      const uint4 pk = pack8(gv);
      *gpp = pk;
      unpack8(pk, gv);
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] += gv[e];
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) sm[pl * chunks * 8 + ck * 8 + e] = a[e];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < nch; c += blockDim.x) {
    float s = 0.f;
    for (int q = 0; q < P; ++q) s += sm[q * chunks * 8 + c];
    part[(size_t)blockIdx.x * nch + c] = s;
  }
}

// ------------------------------------------------------------------------------------------------ resampling
// TF<=1.13 legacy bilinear (align_corners=False, no half-pixel centres): App. A.6.
struct Lerp {
  int lo, hi;
  float f;
};
__device__ __forceinline__ Lerp legacy_lerp(int d, int n_in, float scale) {
  const float s = d * scale;
  Lerp r;
  r.lo = (int)floorf(s);
  r.hi = min(r.lo + 1, n_in - 1);
  r.f = s - (float)r.lo;
  return r;
}
__global__ void resize_bilinear_bf16_kernel(const bf16* __restrict__ src, int sp, int sc, int N, int H, int W, bf16* __restrict__ dst, int dp,
                                            int dc, int OH, int OW, int chunks) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)N * OH * OW * chunks;
  if (i >= total) return;
  const int c = (int)(i % chunks) * 8;
  size_t pix = i / chunks;
  const int ox = (int)(pix % OW);
  const int oy = (int)((pix / OW) % OH);
  const int n = (int)(pix / ((size_t)OW * OH));
  const Lerp ly = legacy_lerp(oy, H, (float)H / (float)OH), lx = legacy_lerp(ox, W, (float)W / (float)OW);
  float tl[8], tr[8], bl[8], br[8], o[8];
  const bf16* b = src + (size_t)n * H * W * sp + sc + c;
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)ly.lo * W + lx.lo) * sp), tl);
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)ly.lo * W + lx.hi) * sp), tr);
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)ly.hi * W + lx.lo) * sp), bl);
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)ly.hi * W + lx.hi) * sp), br);
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float t = tl[e] + (tr[e] - tl[e]) * lx.f;
    const float bo = bl[e] + (br[e] - bl[e]) * lx.f;
    o[e] = t + (bo - t) * ly.f;
  }
  *reinterpret_cast<uint4*>(dst + pix * dp + dc + c) = pack8(o);
}
// weight of source index i in destination index d (transpose of legacy_lerp)
__device__ __forceinline__ float legacy_w(int d, int i, int n_in, float scale) {
  const Lerp l = legacy_lerp(d, n_in, scale);
  return (l.lo == i ? 1.f - l.f : 0.f) + (l.hi == i ? l.f : 0.f);
}
__device__ __forceinline__ void legacy_range(int i, int n_out, float scale, int& d0, int& d1) {
  d0 = max(0, (int)floorf((i - 1) / scale) - 1);
  d1 = min(n_out - 1, (int)ceilf((i + 1) / scale) + 1);
}
__global__ void resize_bilinear_bf16_bwd_kernel(const bf16* __restrict__ dd, int dp, int dc, int N, int OH, int OW, bf16* ds, int sp, int sc,
                                                int H, int W, int chunks, int accumulate) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)N * H * W * chunks;
  if (i >= total) return;
  const int c = (int)(i % chunks) * 8;
  size_t pix = i / chunks;
  const int x = (int)(pix % W);
  const int y = (int)((pix / W) % H);
  const int n = (int)(pix / ((size_t)W * H));
  const float sy = (float)H / (float)OH, sx = (float)W / (float)OW;
  int y0, y1, x0, x1;
  legacy_range(y, OH, sy, y0, y1);
  legacy_range(x, OW, sx, x0, x1);
  float a[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t[8];
  uint4* o = reinterpret_cast<uint4*>(ds + pix * sp + sc + c);
  if (accumulate) unpack8(*o, a);
  for (int dy = y0; dy <= y1; ++dy) {
    const float wy = legacy_w(dy, y, H, sy);
    if (wy == 0.f) continue;
    for (int dx = x0; dx <= x1; ++dx) {
      const float wt = wy * legacy_w(dx, x, W, sx);
      if (wt == 0.f) continue;
      unpack8(*reinterpret_cast<const uint4*>(dd + ((size_t)(n * OH + dy) * OW + dx) * dp + dc + c), t);
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] += wt * t[e];
    }
  }
  *o = pack8(a);
}
// ---- fused resize + concat (recover decoder, convolution_utils.py:87-90 + nets.py:80-105): up to 4 sources of one resolution, each
// a channel slice of its own tensor (batch-broadcast when n_mod > 0), are legacy-bilinear resized to OH x OW and written side by side
// into ONE destination slice -- one launch instead of a resize per source plus a copy per source (and per broadcast replica).
struct RcArgs {
  CisSrc s[CIS_MAX_SRC];
  int nsrc;
};
__global__ void resize_concat_bf16_kernel(const RcArgs a, int N, int H, int W, bf16* __restrict__ dst, int dp, int dc, int OH, int OW,
                                          int total_chunks) {
  // grid.y = destination row (n, oy), grid.x * 256 threads = (ox, 8-channel chunk) of that row: no 64-bit divisions per thread
  pdl_launch_dependents();
  pdl_wait();
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (unsigned)(OW * total_chunks)) return;
  const int ox = (int)(t / (unsigned)total_chunks);
  int ck = (int)(t - (unsigned)ox * (unsigned)total_chunks);
  const int n = (int)(blockIdx.y / (unsigned)OH), oy = (int)(blockIdx.y - (unsigned)n * (unsigned)OH);
  const int off = ck * 8;
  int si = 0;
  while (si < a.nsrc - 1 && ck >= a.s[si].chunks) {
    ck -= a.s[si].chunks;
    ++si;
  }
  CisSrc sd = a.s[0];
  if (si == 1) sd = a.s[1];
  if (si == 2) sd = a.s[2];
  if (si == 3) sd = a.s[3];
  const int ns = sd.n_mod ? n % sd.n_mod : n;
  const bf16* b = reinterpret_cast<const bf16*>(sd.ptr) + (size_t)ns * H * W * sd.pitch + sd.c_off + ck * 8;
  uint4* o = reinterpret_cast<uint4*>(dst + ((size_t)blockIdx.y * OW + ox) * dp + dc + off);
  if (H == OH && W == OW) {          // same resolution: a plain gather of the channel slices
    *o = *reinterpret_cast<const uint4*>(b + ((size_t)oy * W + ox) * sd.pitch);
    return;
  }
  const Lerp ly = legacy_lerp(oy, H, (float)H / (float)OH), lx = legacy_lerp(ox, W, (float)W / (float)OW);
  float tl[8], tr[8], bl[8], br[8], r[8];
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)ly.lo * W + lx.lo) * sd.pitch), tl);
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)ly.lo * W + lx.hi) * sd.pitch), tr);
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)ly.hi * W + lx.lo) * sd.pitch), bl);
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)ly.hi * W + lx.hi) * sd.pitch), br);
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float tp = tl[e] + (tr[e] - tl[e]) * lx.f;
    const float bo = bl[e] + (br[e] - bl[e]) * lx.f;
    r[e] = tp + (bo - tp) * ly.f;
  }
  *o = pack8(r);
}
// exact x2 case (OH = 2H, OW = 2W: every `deconv` of the recover decoder at power-of-two sizes): one thread per SOURCE pixel chunk loads the
// 2x2 source neighbourhood once and writes the four destination pixels it determines -- same lerp expressions (fractions 0 / 0.5, clamped
// last row / column), so the result is bit-identical to the generic kernel with a quarter of the loads and index arithmetic.
__global__ void resize_concat_x2_bf16_kernel(const RcArgs a, int N, int H, int W, bf16* __restrict__ dst, int dp, int dc, int total_chunks) {
  pdl_launch_dependents();
  pdl_wait();
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (unsigned)(W * total_chunks)) return;
  const int x = (int)(t / (unsigned)total_chunks);
  int ck = (int)(t - (unsigned)x * (unsigned)total_chunks);
  const int n = (int)(blockIdx.y / (unsigned)H), y = (int)(blockIdx.y - (unsigned)n * (unsigned)H);
  const int off = ck * 8;
  int si = 0;
  while (si < a.nsrc - 1 && ck >= a.s[si].chunks) {
    ck -= a.s[si].chunks;
    ++si;
  }
  CisSrc sd = a.s[0];
  if (si == 1) sd = a.s[1];
  if (si == 2) sd = a.s[2];
  if (si == 3) sd = a.s[3];
  const int ns = sd.n_mod ? n % sd.n_mod : n;
  const bf16* b = reinterpret_cast<const bf16*>(sd.ptr) + (size_t)ns * H * W * sd.pitch + sd.c_off + ck * 8;
  const int x1 = min(x + 1, W - 1), y1 = min(y + 1, H - 1);
  float s00[8], s01[8], s10[8], s11[8], r[8];
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)y * W + x) * sd.pitch), s00);
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)y * W + x1) * sd.pitch), s01);
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)y1 * W + x) * sd.pitch), s10);
  unpack8(*reinterpret_cast<const uint4*>(b + ((size_t)y1 * W + x1) * sd.pitch), s11);
  const int OW = 2 * W;
  bf16* o = dst + (((size_t)(n * 2 * H + 2 * y)) * OW + 2 * x) * dp + dc + off;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float fy = (q >> 1) ? 0.5f : 0.f, fx = (q & 1) ? 0.5f : 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float tp = s00[e] + (s01[e] - s00[e]) * fx;
      const float bo = s10[e] + (s11[e] - s10[e]) * fx;
      r[e] = tp + (bo - tp) * fy;
    }
    *reinterpret_cast<uint4*>(o + ((size_t)(q >> 1) * OW + (q & 1)) * dp) = pack8(r);
  }
}
// its transpose: for every source with want != 0, dsrc (=|+=) sum over broadcast replicas of R^T ddst[.., slice of that source]
struct RcGrad {
  void* ptr;
  int pitch, c_off, chunks, n_mod, want, accumulate;
};
struct RcGradArgs {
  RcGrad s[CIS_MAX_SRC];
  int nsrc;
};
__global__ void resize_concat_bf16_bwd_kernel(const bf16* __restrict__ dd, int dp, int dc, int N, int OH, int OW, const RcGradArgs a, int H,
                                              int W, int total_chunks) {
  // grid.y = source row (n, y), grid.x * 256 threads = (x, 8-channel chunk).  The x weights of the (<= 8 wide) candidate window are
  // evaluated once per thread, not once per (dy, dx) pair.
  pdl_launch_dependents();
  pdl_wait();
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (unsigned)(W * total_chunks)) return;
  const int x = (int)(t / (unsigned)total_chunks);
  int ck = (int)(t - (unsigned)x * (unsigned)total_chunks);
  const int n = (int)(blockIdx.y / (unsigned)H), y = (int)(blockIdx.y - (unsigned)n * (unsigned)H);
  const int off = ck * 8;
  int si = 0;
  while (si < a.nsrc - 1 && ck >= a.s[si].chunks) {
    ck -= a.s[si].chunks;
    ++si;
  }
  RcGrad sd = a.s[0];
  if (si == 1) sd = a.s[1];
  if (si == 2) sd = a.s[2];
  if (si == 3) sd = a.s[3];
  if (!sd.want || (sd.n_mod && n >= sd.n_mod)) return;
  const int reps = sd.n_mod ? N / sd.n_mod : 1;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tv[8];
  uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(sd.ptr) + ((size_t)(n * H + y) * W + x) * sd.pitch + sd.c_off + ck * 8);
  if (sd.accumulate) unpack8(*o, acc);
  if (H == OH && W == OW) {          // same resolution: fold the broadcast replicas of this pixel
    for (int r = 0; r < reps; ++r) {
      unpack8(*reinterpret_cast<const uint4*>(dd + ((size_t)((n + r * sd.n_mod) * OH + y) * OW + x) * dp + dc + off), tv);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] += tv[e];
    }
    *o = pack8(acc);
    return;
  }
  const float sy = (float)H / (float)OH, sx = (float)W / (float)OW;
  const bool x2 = OH == 2 * H && OW == 2 * W;     // exact x2: the transpose weights are 0.5 / 1 / 0.5 (1 on the clamped last row / column),
  int y0, y1, x0, x1;                             // the same values legacy_w returns, without evaluating it 14 times per thread
  if (x2) {
    y0 = max(2 * y - 1, 0);
    y1 = 2 * y + 1;
    x0 = max(2 * x - 1, 0);
    x1 = 2 * x + 1;
  } else {
    legacy_range(y, OH, sy, y0, y1);
    legacy_range(x, OW, sx, x0, x1);
  }
  const int nx = x1 - x0 + 1;
  const bool pre = nx <= 8;
  float wxv[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int dx = x0 + k;
    wxv[k] = !(pre && k < nx) ? 0.f : x2 ? ((dx == 2 * x || (dx == 2 * x + 1 && x == W - 1)) ? 1.f : 0.5f) : legacy_w(dx, x, W, sx);
  }
  for (int dy = y0; dy <= y1; ++dy) {
    const float wy = x2 ? ((dy == 2 * y || (dy == 2 * y + 1 && y == H - 1)) ? 1.f : 0.5f) : legacy_w(dy, y, H, sy);
    if (wy == 0.f) continue;
    if (pre) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float wt = wy * wxv[k];
        if (wt == 0.f) continue;
        for (int r = 0; r < reps; ++r) {
          unpack8(*reinterpret_cast<const uint4*>(dd + ((size_t)((n + r * sd.n_mod) * OH + dy) * OW + x0 + k) * dp + dc + off), tv);
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[e] += wt * tv[e];
        }
      }
    } else {
      for (int dx = x0; dx <= x1; ++dx) {
        const float wt = wy * legacy_w(dx, x, W, sx);
        if (wt == 0.f) continue;
        for (int r = 0; r < reps; ++r) {
          unpack8(*reinterpret_cast<const uint4*>(dd + ((size_t)((n + r * sd.n_mod) * OH + dy) * OW + dx) * dp + dc + off), tv);
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[e] += wt * tv[e];
        }
      }
    }
  }
  *o = pack8(acc);
}
__global__ void resize_bilinear_f32_kernel(const float* __restrict__ src, int N, int H, int W, int C, float* __restrict__ dst, int OH, int OW,
                                           float scale) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= (size_t)N * OH * OW) return;
  const int ox = (int)(pix % OW);
  const int oy = (int)((pix / OW) % OH);
  const int n = (int)(pix / ((size_t)OW * OH));
  const Lerp ly = legacy_lerp(oy, H, (float)H / (float)OH), lx = legacy_lerp(ox, W, (float)W / (float)OW);
  const float* b = src + (size_t)n * H * W * C;
  for (int c = 0; c < C; ++c) {
    const float tl = b[((size_t)ly.lo * W + lx.lo) * C + c], tr = b[((size_t)ly.lo * W + lx.hi) * C + c];
    const float bl = b[((size_t)ly.hi * W + lx.lo) * C + c], br = b[((size_t)ly.hi * W + lx.hi) * C + c];
    const float t = tl + (tr - tl) * lx.f, bo = bl + (br - bl) * lx.f;
    dst[pix * C + c] = (t + (bo - t) * ly.f) * scale;
  }
}
// central crop + legacy-bilinear resize back to OH x OW of ONE fp32 NHWC image (the multi-crop ensemble inputs,
// davis2016_data_utils.py:328-354 / 130-134): crop box (y0, x0, ch, cw) of the Hs x Ws source, same interpolation rule as above
__global__ void crop_resize_f32_kernel(const float* __restrict__ src, int Ws, int C, int y0, int x0, int ch, int cw, float* __restrict__ dst,
                                       int OH, int OW) {
  pdl_launch_dependents();
  pdl_wait();
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= OH * OW) return;
  const int ox = pix % OW, oy = pix / OW;
  const Lerp ly = legacy_lerp(oy, ch, (float)ch / (float)OH), lx = legacy_lerp(ox, cw, (float)cw / (float)OW);
  const float* r0 = src + (size_t)(y0 + ly.lo) * Ws * C;
  const float* r1 = src + (size_t)(y0 + ly.hi) * Ws * C;
  for (int c = 0; c < C; ++c) {
    const float tl = r0[(x0 + lx.lo) * C + c], tr = r0[(x0 + lx.hi) * C + c];
    const float bl = r1[(x0 + lx.lo) * C + c], br = r1[(x0 + lx.hi) * C + c];
    const float t = tl + (tr - tl) * lx.f, bo = bl + (br - bl) * lx.f;
    dst[(size_t)pix * C + c] = t + (bo - t) * ly.f;
  }
}
// transpose of the fp32 legacy resize, result stored as a bf16 8-channel chunk (C <= 8 real channels)
__global__ void resize_f32_bwd_to_bf16_kernel(const float* __restrict__ dd, int N, int OH, int OW, int C, int H, int W, bf16* __restrict__ ds,
                                              int sp) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= (size_t)N * H * W) return;
  const int x = (int)(pix % W);
  const int y = (int)((pix / W) % H);
  const int n = (int)(pix / ((size_t)W * H));
  const float sy = (float)H / (float)OH, sx = (float)W / (float)OW;
  int y0, y1, x0, x1;
  legacy_range(y, OH, sy, y0, y1);
  legacy_range(x, OW, sx, x0, x1);
  float a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int dy = y0; dy <= y1; ++dy) {
    const float wy = legacy_w(dy, y, H, sy);
    if (wy == 0.f) continue;
    for (int dx = x0; dx <= x1; ++dx) {
      const float wt = wy * legacy_w(dx, x, W, sx);
      if (wt == 0.f) continue;
      const float* q = dd + ((size_t)(n * OH + dy) * OW + dx) * C;
      for (int c = 0; c < C; ++c) a[c] += wt * q[c];
    }
  }
  *reinterpret_cast<uint4*>(ds + pix * sp) = pack8(a);
}
// tf.image.resize_nearest_neighbor(align_corners=True), out = 2*in: src = min(roundf(d*(in-1)/(out-1)), in-1)   App. A.5
__device__ __forceinline__ int nn_src(int d, int n_in) {
  const float scale = (float)(n_in - 1) / (float)(2 * n_in - 1);
  return min((int)roundf(d * scale), n_in - 1);
}
__global__ void upsample_nn2x_kernel(const bf16* __restrict__ src, int N, int H, int W, int pitch, bf16* __restrict__ dst) {
  // grid.y = destination row (n, oy); threads = (ox, 8-channel chunk): 32-bit index math, one source row per block row
  pdl_launch_dependents();
  pdl_wait();
  const int chunks = pitch / 8;
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (unsigned)(2 * W * chunks)) return;
  const int ox = (int)(t / (unsigned)chunks), c = (int)(t - (unsigned)ox * (unsigned)chunks) * 8;
  const int n = (int)(blockIdx.y / (unsigned)(2 * H)), oy = (int)(blockIdx.y - (unsigned)n * (unsigned)(2 * H));
  const int sy = nn_src(oy, H), sx = nn_src(ox, W);
  *reinterpret_cast<uint4*>(dst + ((size_t)blockIdx.y * 2 * W + ox) * pitch + c) =
      *reinterpret_cast<const uint4*>(src + ((size_t)(n * H + sy) * W + sx) * pitch + c);
}
__global__ void upsample_nn2x_bwd_kernel(const bf16* __restrict__ dd, int N, int H, int W, int pitch, bf16* ds, int accumulate) {
  // grid.y = source row (n, y); the (<= 6) candidate destination rows / columns are tested once per thread, not once per pair
  pdl_launch_dependents();
  pdl_wait();
  const int chunks = pitch / 8;
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (unsigned)(W * chunks)) return;
  const int x = (int)(t / (unsigned)chunks), c = (int)(t - (unsigned)x * (unsigned)chunks) * 8;
  const int n = (int)(blockIdx.y / (unsigned)H), y = (int)(blockIdx.y - (unsigned)n * (unsigned)H);
  float a[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tv[8];
  uint4* o = reinterpret_cast<uint4*>(ds + ((size_t)blockIdx.y * W + x) * pitch + c);
  if (accumulate) unpack8(*o, a);
  const int dx0 = max(0, 2 * x - 2), dx1 = min(2 * W - 1, 2 * x + 3);
  unsigned xm = 0;                                   // bit k: destination column dx0 + k maps to this source column
  for (int dx = dx0; dx <= dx1; ++dx)
    if (nn_src(dx, W) == x) xm |= 1u << (dx - dx0);
  for (int dy = max(0, 2 * y - 2); dy <= min(2 * H - 1, 2 * y + 3); ++dy) {
    if (nn_src(dy, H) != y) continue;
    const bf16* row = dd + ((size_t)(n * 2 * H + dy) * 2 * W) * pitch + c;
    for (int dx = dx0; dx <= dx1; ++dx) {
      if (!((xm >> (dx - dx0)) & 1u)) continue;
      unpack8(*reinterpret_cast<const uint4*>(row + (size_t)dx * pitch), tv);
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] += tv[e];
    }
  }
  *o = pack8(a);
}
__global__ void resize_nn_f32_kernel(const float* __restrict__ src, int N, int H, int W, int C, float* __restrict__ dst, int OH, int OW) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= (size_t)N * OH * OW) return;
  const int ox = (int)(pix % OW);
  const int oy = (int)((pix / OW) % OH);
  const int n = (int)(pix / ((size_t)OW * OH));
  const int sy = min((int)floorf(oy * ((float)H / (float)OH)), H - 1), sx = min((int)floorf(ox * ((float)W / (float)OW)), W - 1);
  for (int c = 0; c < C; ++c) dst[pix * C + c] = src[((size_t)(n * H + sy) * W + sx) * C + c];
}

// ------------------------------------------------------------------------------------------------ warp + cost volume
// dense_image_warp (core_warp.py:153-202): query = grid - flow, floor clamped to [0,size-2], alpha clamped to [0,1].
__device__ __forceinline__ void warp_coords(float q, int size, int& lo, float& a) {
  float fl = fminf(fmaxf(floorf(q), 0.f), (float)(size - 2));
  lo = (int)fl;
  a = fminf(fmaxf(q - fl, 0.f), 1.f);
}
__device__ __forceinline__ void warp_chunk(const bf16* __restrict__ img, int pitch, int h, int w, int b, float qy, float qx, float* o) {
  int y0, x0;
  float ay, ax;
  warp_coords(qy, h, y0, ay);
  warp_coords(qx, w, x0, ax);
  const bf16* base = img + ((size_t)(b * h + y0) * w + x0) * pitch;
  float tl[8], tr[8], bl[8], br[8];
  unpack8(__ldg(reinterpret_cast<const uint4*>(base)), tl);
  unpack8(__ldg(reinterpret_cast<const uint4*>(base + pitch)), tr);
  unpack8(__ldg(reinterpret_cast<const uint4*>(base + (size_t)w * pitch)), bl);
  unpack8(__ldg(reinterpret_cast<const uint4*>(base + (size_t)w * pitch + pitch)), br);
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float t = ax * (tr[e] - tl[e]) + tl[e];
    const float bo = ax * (br[e] - bl[e]) + bl[e];
    o[e] = ay * (bo - t) + t;
  }
}
__global__ void dense_image_warp_kernel(const bf16* __restrict__ img, int pitch, int coff, const float* __restrict__ flow, float fs, int B,
                                        int h, int w, int chunks, bf16* __restrict__ out, int op) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * h * w * chunks) return;
  const int c = (int)(i % chunks) * 8;
  const size_t pix = i / chunks;
  const int x = (int)(pix % w), y = (int)((pix / w) % h), b = (int)(pix / ((size_t)w * h));
  float o[8];
  warp_chunk(img + coff + c, pitch, h, w, b, (float)y - flow[pix * 2] * fs, (float)x - flow[pix * 2 + 1] * fs, o);
  *reinterpret_cast<uint4*>(out + pix * op + c) = pack8(o);
}

static constexpr int kCvTH = 8, kCvTW = 16, kCvR = 4;
static constexpr int kCvHH = kCvTH + 2 * kCvR, kCvHW = kCvTW + 2 * kCvR;  // 16 x 24 halo
static constexpr int kCvPitch = 36;                                        // floats per smem pixel row (32 ch + pad)
static constexpr int kCvSmem = (kCvTH * kCvTW + kCvHH * kCvHW) * kCvPitch * 4;

__global__ void __launch_bounds__(256) warp_costvol_kernel(const bf16* __restrict__ c1, int c1p, int c1o, const bf16* __restrict__ c2, int c2p,
                                                           int c2o, const float* __restrict__ flow, float fs, int B, int h, int w, int C,
                                                           bf16* __restrict__ out, int op, int oo) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float cvs[];
  float* s1 = cvs;                                 // [128][36]
  float* s2 = cvs + kCvTH * kCvTW * kCvPitch;      // [384][36]
  const int tid = threadIdx.x;
  const int b = blockIdx.z, y0 = blockIdx.y * kCvTH, x0 = blockIdx.x * kCvTW;
  const int pix = tid & 127, py = pix >> 4, px = pix & 15;
  const int dyb = tid >> 7;  // this thread handles dy = dyb + 2k
  float acc[5][9];
#pragma unroll
  for (int k = 0; k < 5; ++k)
#pragma unroll
    for (int d = 0; d < 9; ++d) acc[k][d] = 0.f;
  const int Cp = (C + 7) & ~7;
  for (int cc = 0; cc < Cp; cc += 32) {
    const int nck = min(4, (Cp - cc) / 8);  // 8-channel chunks in this pass
    // c1 tile
    for (int it = tid; it < 128 * 4; it += 256) {
      const int p = it >> 2, ck = it & 3;
      const int y = y0 + (p >> 4), x = x0 + (p & 15);
      float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (ck < nck && y < h && x < w) unpack8(__ldg(reinterpret_cast<const uint4*>(c1 + ((size_t)(b * h + y) * w + x) * c1p + c1o + cc + ck * 8)), v);
      float4* d = reinterpret_cast<float4*>(s1 + p * kCvPitch + ck * 8);
      d[0] = make_float4(v[0], v[1], v[2], v[3]);
      d[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
    // warped c2 halo (zero outside the image: tf.pad of the warped map, core_costvol.py:27)
    for (int it = tid; it < kCvHH * kCvHW * 4; it += 256) {
      const int p = it >> 2, ck = it & 3;
      const int y = y0 - kCvR + p / kCvHW, x = x0 - kCvR + p % kCvHW;
      float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (ck < nck && y >= 0 && y < h && x >= 0 && x < w) {
        if (flow) {
          const size_t fp = ((size_t)(b * h + y) * w + x) * 2;
          warp_chunk(c2 + c2o + cc + ck * 8, c2p, h, w, b, (float)y - __ldg(flow + fp) * fs, (float)x - __ldg(flow + fp + 1) * fs, v);
        } else {
          unpack8(__ldg(reinterpret_cast<const uint4*>(c2 + ((size_t)(b * h + y) * w + x) * c2p + c2o + cc + ck * 8)), v);
        }
      }
      float4* d = reinterpret_cast<float4*>(s2 + p * kCvPitch + ck * 8);
      d[0] = make_float4(v[0], v[1], v[2], v[3]);
      d[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const int dy = dyb + 2 * k;
      if (dy < 9) {
        const float* r2 = s2 + ((py + dy) * kCvHW + px) * kCvPitch;
        const float* r1 = s1 + pix * kCvPitch;
        for (int c4 = 0; c4 < nck * 2; ++c4) {
          const float4 a = *reinterpret_cast<const float4*>(r1 + c4 * 4);
#pragma unroll
          for (int dx = 0; dx < 9; ++dx) {
            const float4 q = *reinterpret_cast<const float4*>(r2 + dx * kCvPitch + c4 * 4);
            acc[k][dx] += a.x * q.x + a.y * q.y + a.z * q.z + a.w * q.w;
          }
        }
      }
    }
    __syncthreads();
  }
  // mean over the REAL channel count, leaky 0.1, stage [128][81] bf16 in smem, coalesced store
  bf16* so = reinterpret_cast<bf16*>(s2);
  const float inv = 1.f / (float)C;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    const int dy = dyb + 2 * k;
    if (dy < 9) {
#pragma unroll
      for (int dx = 0; dx < 9; ++dx) {
        float v = acc[k][dx] * inv;
        v = v > 0.f ? v : 0.1f * v;
        so[pix * 81 + dy * 9 + dx] = __float2bfloat16(v);
      }
    }
  }
  __syncthreads();
  for (int it = tid; it < 128 * 81; it += 256) {
    const int p = it / 81, ch = it % 81;
    const int y = y0 + (p >> 4), x = x0 + (p & 15);
    if (y < h && x < w) out[((size_t)(b * h + y) * w + x) * op + oo + ch] = so[it];
  }
}

// ------------------------------------------------------------------------------------------------ input packing
__global__ void pack_f32_to_bf16_kernel(const float* __restrict__ src, size_t npix, int C, float offset, bf16* __restrict__ dst, int dp, int dc) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= npix) return;
  float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int c = 0; c < C; ++c) v[c] = src[pix * C + c] + offset;
  *reinterpret_cast<uint4*>(dst + pix * dp + dc) = pack8(v);
}
__global__ void flow_stats_kernel(const float* __restrict__ flow, size_t hw, double* __restrict__ stats) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.y;
  double s0 = 0, s1 = 0, q0 = 0, q1 = 0;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < hw; p += (size_t)gridDim.x * blockDim.x) {
    const float2 f = *reinterpret_cast<const float2*>(flow + ((size_t)b * hw + p) * 2);
    s0 += f.x; s1 += f.y; q0 += (double)f.x * f.x; q1 += (double)f.y * f.y;
  }
  s0 = warp_sum_d(s0); s1 = warp_sum_d(s1); q0 = warp_sum_d(q0); q1 = warp_sum_d(q1);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(stats + b * 4 + 0, s0); atomicAdd(stats + b * 4 + 1, s1);
    atomicAdd(stats + b * 4 + 2, q0); atomicAdd(stats + b * 4 + 3, q1);
  }
}
__global__ void pack_generator_input_kernel(const float* __restrict__ image, const float* __restrict__ flow, const double* __restrict__ stats,
                                            size_t hw, bf16* __restrict__ dst) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.y;
  const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= hw) return;
  const double n = (double)hw;
  const double m0 = stats[b * 4] / n, m1 = stats[b * 4 + 1] / n;
  const float r0 = (float)(1.0 / sqrt(stats[b * 4 + 2] / n - m0 * m0)), r1 = (float)(1.0 / sqrt(stats[b * 4 + 3] / n - m1 * m1));
  const size_t pix = (size_t)b * hw + p;
  float v[8] = {image[pix * 3], image[pix * 3 + 1], image[pix * 3 + 2], (flow[pix * 2] - (float)m0) * r0, (flow[pix * 2 + 1] - (float)m1) * r1,
                0, 0, 0};
  *reinterpret_cast<uint4*>(dst + pix * 8) = pack8(v);
}

// ------------------------------------------------------------------------------------------------ mask (x) flow + loss
__global__ void mask_apply_kernel(const float* __restrict__ flow, const float* __restrict__ mask, size_t npix, bf16* __restrict__ dst) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npix) return;
  const float m = mask[p], f0 = flow[p * 2], f1 = flow[p * 2 + 1];
  const float a[8] = {f0 * (1.f - m), f1 * (1.f - m), 1.f, 1.f - m, 0, 0, 0, 0};  // adversarial_learner.py:109 + nets.py:50-52
  const float c[8] = {f0 * m, f1 * m, 1.f, m, 0, 0, 0, 0};                          // :110 with mask = 1-m
  const float z[8] = {0, 0, 1.f, 0, 0, 0, 0, 0};                                    // :127-131
  *reinterpret_cast<uint4*>(dst + p * 8) = pack8(a);
  *reinterpret_cast<uint4*>(dst + (npix + p) * 8) = pack8(c);
  *reinterpret_cast<uint4*>(dst + (2 * npix + p) * 8) = pack8(z);
}
__device__ __forceinline__ float2 pred_at(const float* __restrict__ f1, int n, int h1, int w1, const Lerp& ly, const Lerp& lx) {
  const float2* b = reinterpret_cast<const float2*>(f1) + (size_t)n * h1 * w1;
  const float2 tl = b[(size_t)ly.lo * w1 + lx.lo], tr = b[(size_t)ly.lo * w1 + lx.hi];
  const float2 bl = b[(size_t)ly.hi * w1 + lx.lo], br = b[(size_t)ly.hi * w1 + lx.hi];
  float2 r;
  {
    const float t = tl.x + (tr.x - tl.x) * lx.f, bo = bl.x + (br.x - bl.x) * lx.f;
    r.x = t + (bo - t) * ly.f;
  }
  {
    const float t = tl.y + (tr.y - tl.y) * lx.f, bo = bl.y + (br.y - bl.y) * lx.f;
    r.y = t + (bo - t) * ly.f;
  }
  return r;
}
// charbonnier term (loss_utils.py:47-49) and its derivative w.r.t. pred
__device__ __forceinline__ float charb(float d, float cbn) {
  const float s = d * d + 1e-6f;
  return cbn == 0.5f ? sqrtf(s) : powf(s, cbn);
}
__device__ __forceinline__ float dcharb_dpred(float d, float cbn) {  // d = gt - pred
  const float s = d * d + 1e-6f;
  return cbn == 0.5f ? -d * rsqrtf(s) : -2.f * cbn * d * powf(s, cbn - 1.f);
}
// Stand-alone charbonnier_loss (loss_utils.py:34-51) for the functional API: sums[b] = sum_{p,c} ((gt-pred)^2 + 1e-6)^cbn * mask.
// mask_c = 1: one mask value per pixel (broadcast over the C channels), mask_c = C: one per element.  sums (double) must be zeroed.
__global__ void charbonnier_sum_kernel(const float* __restrict__ gt, const float* __restrict__ pred, const float* __restrict__ mask, size_t hw,
                                       int C, int mask_c, float cbn, double* __restrict__ sums) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.y;
  double acc = 0;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < hw; p += (size_t)gridDim.x * blockDim.x) {
    const size_t base = ((size_t)b * hw + p);
    for (int c = 0; c < C; ++c) {
      const float m = mask[mask_c == 1 ? base : base * C + c];
      acc += (double)(charb(gt[base * C + c] - pred[base * C + c], cbn) * m);
    }
  }
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) atomicAdd(sums + b, acc);
}
__global__ void cis_loss_fwd_kernel(const float* __restrict__ flow, const float* __restrict__ mask, const float* __restrict__ flow1, int B, int H,
                                    int W, int h1, int w1, float cbn, double* __restrict__ sums, float* __restrict__ pred_out) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.y;
  const size_t hw = (size_t)H * W;
  float a[5] = {0, 0, 0, 0, 0};
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < hw; p += (size_t)gridDim.x * blockDim.x) {
    const int y = (int)(p / W), x = (int)(p % W);
    const Lerp ly = legacy_lerp(y, h1, (float)h1 / (float)H), lx = legacy_lerp(x, w1, (float)w1 / (float)W);
    const size_t pix = (size_t)b * hw + p;
    const float m = mask[pix];
    const float2 f = *reinterpret_cast<const float2*>(flow + pix * 2);
    float e[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const float2 pr = pred_at(flow1, j * B + b, h1, w1, ly, lx);
      e[j] = charb(f.x - pr.x, cbn) + charb(f.y - pr.y, cbn);
      if (pred_out) *reinterpret_cast<float2*>(pred_out + ((size_t)(j * B + b) * hw + p) * 2) = pr;
    }
    a[0] += m * e[0];           // rec           adversarial_learner.py:144
    a[1] += (1.f - m) * e[1];   // rec_compl     :149
    a[2] += e[2];               // image prior   :161
    a[3] += m * e[2];           // den_red       :179
    a[4] += (1.f - m) * e[2];   // den_red_compl :186
  }
  // block-level reduction first: one fp64 atomic per (block, sum) instead of one per warp -- 23.7 k atomics on 20 addresses serialised
  // in L2 for ~25 us of this kernel's 31 us, between the forward and the backward pass of every step
  __shared__ float red[8][5];
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    const float s = warp_sum(a[k]);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][k] = s;
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += (double)red[w][threadIdx.x];
    atomicAdd(sums + b * 5 + threadIdx.x, t);
  }
}
__global__ void cis_loss_reduce_kernel(const double* __restrict__ sums, int B, int GB, double hw, float eps, float* __restrict__ scalars,
                                       float* __restrict__ coef) {
  pdl_launch_dependents();
  pdl_wait();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double rec_total = 0, rr = 0, rrc = 0;
  for (int b = 0; b < B; ++b) {
    const double rec = sums[b * 5], recc = sums[b * 5 + 1], prior = sums[b * 5 + 2];
    const double D = sums[b * 5 + 3] + eps, Dc = sums[b * 5 + 4] + eps;
    rec_total += rec + recc + prior;
    rr += 1.0 - rec / D;
    rrc += 1.0 - recc / Dc;
    coef[b * 4 + 0] = (float)(-1.0 / (GB * D));
    coef[b * 4 + 1] = (float)(rec / (GB * D * D));
    coef[b * 4 + 2] = (float)(-1.0 / (GB * Dc));
    coef[b * 4 + 3] = (float)(recc / (GB * Dc * Dc));
  }
  scalars[2] = (float)(rr / GB);
  scalars[3] = (float)(rrc / GB);
  scalars[0] = scalars[2] + scalars[3];                  // generator loss  :194
  scalars[1] = (float)(rec_total / (hw * (double)GB));   // recover loss    :171-172
  scalars[4] = (float)(1.0 / (hw * (double)GB));
}
__global__ void cis_loss_bwd_kernel(const float* __restrict__ flow, const float* __restrict__ mask, const float* __restrict__ flow1,
                                    const float* __restrict__ coef, const float* __restrict__ scalars, int B, int H, int W, int h1, int w1,
                                    float cbn, int which, float* __restrict__ dpred, float* __restrict__ dmask) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.y;
  const size_t hw = (size_t)H * W;
  const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= hw) return;
  const int y = (int)(p / W), x = (int)(p % W);
  const Lerp ly = legacy_lerp(y, h1, (float)h1 / (float)H), lx = legacy_lerp(x, w1, (float)w1 / (float)W);
  const size_t pix = (size_t)b * hw + p;
  const float m = mask[pix];
  const float2 f = *reinterpret_cast<const float2*>(flow + pix * 2);
  float2 pr[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) pr[j] = pred_at(flow1, j * B + b, h1, w1, ly, lx);
  float w0, w1c, w2;
  if (which == 0) {
    const float k = scalars[4];
    w0 = k * m; w1c = k * (1.f - m); w2 = k;
  } else {
    const float a = coef[b * 4], c = coef[b * 4 + 1], ac = coef[b * 4 + 2], ccq = coef[b * 4 + 3];
    w0 = a * m; w1c = ac * (1.f - m); w2 = c * m + ccq * (1.f - m);
    const float e0 = charb(f.x - pr[0].x, cbn) + charb(f.y - pr[0].y, cbn);
    const float e1 = charb(f.x - pr[1].x, cbn) + charb(f.y - pr[1].y, cbn);
    const float e2 = charb(f.x - pr[2].x, cbn) + charb(f.y - pr[2].y, cbn);
    dmask[pix] = a * e0 - ac * e1 + (c - ccq) * e2;
  }
  const float wj[3] = {w0, w1c, w2};
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    float2 g;
    g.x = wj[j] * dcharb_dpred(f.x - pr[j].x, cbn);
    g.y = wj[j] * dcharb_dpred(f.y - pr[j].y, cbn);
    *reinterpret_cast<float2*>(dpred + ((size_t)(j * B + b) * hw + p) * 2) = g;
  }
}
__global__ void mask_bwd_kernel(const float* __restrict__ flow, const float* __restrict__ mask, const float* __restrict__ dmd,
                                const bf16* __restrict__ din, size_t npix, bf16* __restrict__ dlogits) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npix) return;
  const float m = mask[p], f0 = flow[p * 2], f1 = flow[p * 2 + 1];
  float d0[8], d1[8];
  unpack8(*reinterpret_cast<const uint4*>(din + p * 8), d0);            // call 0 inputs [f(1-m), 1, 1-m]
  unpack8(*reinterpret_cast<const uint4*>(din + (npix + p) * 8), d1);   // call 1 inputs [f m, 1, m]
  float dm = dmd[p];
  dm += -(f0 * d0[0] + f1 * d0[1]) - d0[3];
  dm += (f0 * d1[0] + f1 * d1[1]) + d1[3];
  const float dl = dm * m * (1.f - m) * 0.1f;  // m = sigmoid((l0-l1)/10)   nets.py:38-41
  const float v[8] = {dl, -dl, 0, 0, 0, 0, 0, 0};
  *reinterpret_cast<uint4*>(dlogits + p * 8) = pack8(v);
}

// ------------------------------------------------------------------------------------------------ optimiser
__global__ void grad_avg_abs_kernel(const float* __restrict__ g, const long long* __restrict__ seg, int nseg, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  // grid = (variables, kAvgAbsChunks): a variable of 2.4 M elements walked by ONE block took 82 us (r02 launch list) -- on the critical
  // path between the backward pass and the optimiser of every generator step
  const int s = blockIdx.x;
  const long long a = seg[2 * s], e = seg[2 * s + 1];
  const long long per = (e - a + gridDim.y - 1) / gridDim.y;
  const long long lo = a + per * blockIdx.y, hi = lo + per < e ? lo + per : e;
  float acc = 0.f;
  for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) acc += fabsf(g[i]);
  __shared__ float red[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(out, v / (float)(e - a) / (float)nseg);  // mean over variables of mean|g|  loss_utils.py:19-20
  }
}
__device__ __forceinline__ uint32_t hash32(uint64_t x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
  return (uint32_t)x;
}
__global__ void clip_adam_kernel(float* __restrict__ param, float* __restrict__ m, float* __restrict__ v, const float* __restrict__ grad, size_t n,
                                 float gscale, float clip, float lr, float b1, float b2, float eps, const long long* __restrict__ step,
                                 const float* __restrict__ avg_abs, int can_change, unsigned long long seed) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long t = step[0] + 1;
  float g = grad[i] * gscale;
  if (can_change && avg_abs[0] < 1e-5f) {
    const uint32_t r = hash32(seed ^ ((uint64_t)t << 40) ^ (uint64_t)i);
    g = fabsf((((float)r + 0.5f) * (1.f / 4294967296.f)) * 2.f * clip - clip);  // |U(-clip, clip)|   loss_utils.py:7-10,23
  } else {
    g = fminf(fmaxf(g, -clip), clip);                                            // loss_utils.py:4-5
  }
  const float lr_t = lr * sqrtf(1.f - powf(b2, (float)t)) / (1.f - powf(b1, (float)t));  // TF Adam (App. A.14)
  const float mi = b1 * m[i] + (1.f - b1) * g;
  const float vi = b2 * v[i] + (1.f - b2) * g * g;
  m[i] = mi;
  v[i] = vi;
  param[i] -= lr_t * mi / (sqrtf(vi) + eps);
}
__global__ void step_inc_kernel(long long* step) {
  pdl_launch_dependents();
  pdl_wait(); step[0] += 1; }
__global__ void abs_sum_kernel(const float* __restrict__ g, size_t n, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  float acc = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) acc += fabsf(g[i]);
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}
__global__ void cast_f32_bf16_kernel(const float* __restrict__ s, size_t n, bf16* __restrict__ d) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d[i] = __float2bfloat16(s[i]);
}
__global__ void cast_bf16_f32_kernel(const bf16* __restrict__ s, size_t npix, int pitch, int coff, int C, float* __restrict__ d) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix * C) return;
  const size_t p = i / C;
  const int c = (int)(i % C);
  d[i] = __bfloat162float(s[p * pitch + coff + c]);
}

}  // namespace cis

using namespace cis;
#include <stdlib.h>
#include <string.h>

// every kernel here starts with griddepcontrol.launch_dependents + griddepcontrol.wait, so it may be launched with programmatic
// stream serialization: its CTAs are scheduled while the previous kernel drains (CIS_PDL=0 turns the attribute off).
static bool misc_pdl_enabled() {
  static const bool on = !(getenv("CIS_PDL") && atoi(getenv("CIS_PDL")) == 0);
  return on;
}
template <typename... KArgs, typename... Args>
static void cis_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
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
  cfg.numAttrs = misc_pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
#define CIS_LAUNCH(kern, grid, block, smem, st, ...) cis_launch(kern, dim3(grid), dim3(block), (size_t)(smem), st, __VA_ARGS__)
#define ST ((cudaStream_t)stream)
static inline unsigned nblk(size_t n, int t = 256) { return (unsigned)((n + t - 1) / t); }
typedef const __nv_bfloat16* cbf;
typedef __nv_bfloat16* mbf;

extern "C" {

int cis_pack_weights(const float* w, const int32_t* kmap, int32_t K_pad, int32_t rows, int32_t cout, int32_t sn, const int32_t* nmap, void* wp,
                     cis_stream_t stream) {
  CIS_LAUNCH(pack_weights_kernel, nblk((size_t)rows * K_pad), 256, 0, ST, w, kmap, K_pad, rows, cout, sn, nmap, (mbf)wp);
  return cis_check_launch("pack_weights");
}
int cis_pack_weights_tiled(const float* w, const int32_t* kmap, int32_t cin8, int32_t ntaps, int32_t n_tiles, int32_t BN, int32_t cout, int32_t sn,
                           const int32_t* nmap, void* out, int32_t layout, cis_stream_t stream) {
  if (layout && cin8 != 16) return cis_set_error(CIS_ERR_BAD_ARG, "cis_pack_weights_tiled: layout 1 packs 16 K positions per tile");
  const size_t total = (size_t)n_tiles * ((cin8 + 63) / 64) * ntaps * BN * 64;
  const unsigned blocks = sn == 1 ? (unsigned)(n_tiles * ((cin8 + 63) / 64) * ntaps) : nblk(total);
  if (BN > 128) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_pack_weights_tiled: BN > 128");
  CIS_LAUNCH(pack_weights_tiled_kernel, blocks, 256, 0, ST, w, kmap, cin8, ntaps, n_tiles, BN, cout, sn, nmap, (mbf)out, layout);
  return cis_check_launch("pack_weights_tiled");
}
int cis_unpack_wgrad(const float* dwp, const int32_t* kmap, int32_t K_pad, int32_t cout, int32_t nsplit, float* dw, const float* colpart,
                     int32_t nblocks, int32_t nch, float* db, int32_t layout, cis_stream_t stream) {
  if (nsplit < 1 || (colpart && (nblocks < 1 || !db)) || (layout != 0 && layout != 1) || K_pad % 4)
    return cis_set_error(CIS_ERR_BAD_ARG, "cis_unpack_wgrad: bad split / column-sum / layout arguments");
  CIS_LAUNCH(unpack_wgrad_kernel, nblk((size_t)cout * K_pad + (colpart ? nch : 0)), 256, 0, ST, dwp, kmap, K_pad, cout, nsplit, dw, colpart, nblocks,
             nch, db, layout);
  return cis_check_launch("unpack_wgrad");
}
int cis_param_multi(const CisParamJob* jobs_dev, int32_t njobs, int32_t total_blocks, cis_stream_t stream) {
  if (!jobs_dev || njobs < 1 || total_blocks < 1) return cis_set_error(CIS_ERR_BAD_ARG, "cis_param_multi: bad job table");
  CIS_LAUNCH(param_multi_kernel, (unsigned)total_blocks, 256, 0, ST, jobs_dev, njobs);
  return cis_check_launch("param_multi");
}
int cis_bn_fold(const float* w, const float* bias, const float* gamma, const float* beta, int64_t nw, int32_t cout, float* w_eff, float* b_eff,
                cis_stream_t stream) {
  CIS_LAUNCH(bn_fold_kernel, nblk((size_t)nw), 256, 0, ST, w, bias, gamma, beta, (size_t)nw, cout, w_eff, b_eff);
  return cis_check_launch("bn_fold");
}
int cis_bn_chain(const float* w, const float* bias, const float* gamma, float* dwe, const float* dbe, int64_t nw, int32_t cout, float* dbias,
                 float* dgamma, float* dbeta, cis_stream_t stream) {
  CIS_LAUNCH(bn_chain_kernel, (unsigned)((cout + kBnChainCo - 1) / kBnChainCo), 256, 0, ST, w, bias, gamma, dwe, dbe, (size_t)nw, cout, dbias, dgamma, dbeta);
  return cis_check_launch("bn_chain");
}
int cis_dact_mul(void* g, int32_t gp, int32_t gc, const void* y, int32_t yp, int32_t yc, const void* res, int32_t rp, int32_t rc, int64_t npix,
                 int32_t chunks, int32_t act, float alpha, cis_stream_t stream) {
  if (act == CIS_ACT_NONE) return CIS_OK;
  CIS_LAUNCH(dact_mul_kernel, nblk((size_t)npix * chunks), 256, 0, ST, (mbf)g, gp, gc, (cbf)y, yp, yc, (cbf)res, rp, rc, (size_t)npix, chunks, act, alpha);
  return cis_check_launch("dact_mul");
}
int cis_add_slice(void* dst, int32_t dp, int32_t dc, const void* src, int32_t sp, int32_t sc, int64_t npix, int32_t chunks, int32_t reps,
                  int32_t accumulate, cis_stream_t stream) {
  CIS_LAUNCH(add_slice_kernel, nblk((size_t)npix * chunks), 256, 0, ST, (mbf)dst, dp, dc, (cbf)src, sp, sc, (size_t)npix, chunks, reps, accumulate);
  return cis_check_launch("add_slice");
}
int cis_colsum(const void* g, int32_t gp, int32_t gc, int64_t npix, int32_t nch, float* part, int32_t nblocks, cis_stream_t stream) {
  const int chunks = (nch + 7) / 8;
  if (chunks > 32) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_colsum: more than 256 channels");
  if (nblocks < 1 || nblocks > 592) return cis_set_error(CIS_ERR_BAD_ARG, "cis_colsum: nblocks must be in [1, 592]");
  const int P = 256 / chunks;
  CIS_LAUNCH(colsum_kernel, (unsigned)nblocks, 256, P * chunks * 8 * sizeof(float), ST, (cbf)g, gp, gc, (size_t)npix, nch, chunks, part);
  return cis_check_launch("colsum");
}
int cis_zero(void* ptr, int64_t nbytes, cis_stream_t stream) {
  if (!ptr || nbytes < 0) return cis_set_error(CIS_ERR_BAD_ARG, "cis_zero: bad buffer");
  cudaError_t e = cudaMemsetAsync(ptr, 0, (size_t)nbytes, ST);     // a memset node under graph capture: no kernel, no library launch
  if (e != cudaSuccess) return cis_set_cuda_error(e, "cudaMemsetAsync");
  return CIS_OK;
}
int cis_dact_colsum(void* g, int32_t gp, int32_t gc, const void* y, int32_t yp, int32_t yc, const void* res, int32_t rp, int32_t rc, int64_t npix,
                    int32_t nch, int32_t act, float alpha, float* part, int32_t nblocks, cis_stream_t stream) {
  const int chunks = (nch + 7) / 8;
  if (act == CIS_ACT_NONE) return cis_colsum(g, gp, gc, npix, nch, part, nblocks, stream);
  if (chunks > 32) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_dact_colsum: more than 256 channels");
  if (nblocks < 1 || nblocks > 592) return cis_set_error(CIS_ERR_BAD_ARG, "cis_dact_colsum: nblocks must be in [1, 592]");
  const int P = 256 / chunks;
  CIS_LAUNCH(dact_colsum_kernel, (unsigned)nblocks, 256, P * chunks * 8 * sizeof(float), ST, (mbf)g, gp, gc, (cbf)y, yp, yc, (cbf)res, rp, rc,
             (size_t)npix, nch, chunks, act, alpha, part);
  return cis_check_launch("dact_colsum");
}
int cis_resize_bilinear_bf16(const void* src, int32_t sp, int32_t sc, int32_t N, int32_t H, int32_t W, void* dst, int32_t dp, int32_t dc, int32_t OH,
                             int32_t OW, int32_t chunks, cis_stream_t stream) {
  CIS_LAUNCH(resize_bilinear_bf16_kernel, nblk((size_t)N * OH * OW * chunks), 256, 0, ST, (cbf)src, sp, sc, N, H, W, (mbf)dst, dp, dc, OH, OW, chunks);
  return cis_check_launch("resize_bilinear_bf16");
}
int cis_resize_bilinear_bf16_bwd(const void* dd, int32_t dp, int32_t dc, int32_t N, int32_t OH, int32_t OW, void* ds, int32_t sp, int32_t sc, int32_t H,
                                 int32_t W, int32_t chunks, int32_t accumulate, cis_stream_t stream) {
  CIS_LAUNCH(resize_bilinear_bf16_bwd_kernel, nblk((size_t)N * H * W * chunks), 256, 0, ST, (cbf)dd, dp, dc, N, OH, OW, (mbf)ds, sp, sc, H, W, chunks,
                                                                                     accumulate);
  return cis_check_launch("resize_bilinear_bf16_bwd");
}
int cis_resize_concat_bf16(const CisSrc* srcs, int32_t nsrc, int32_t N, int32_t H, int32_t W, void* dst, int32_t dp, int32_t dc, int32_t OH, int32_t OW,
                           cis_stream_t stream) {
  if (!srcs || nsrc < 1 || nsrc > CIS_MAX_SRC) return cis_set_error(CIS_ERR_BAD_ARG, "cis_resize_concat_bf16: 1..4 sources");
  RcArgs a;
  a.nsrc = nsrc;
  int total = 0;
  for (int i = 0; i < nsrc; ++i) {
    a.s[i] = srcs[i];
    if ((srcs[i].pitch | srcs[i].c_off) & 7) return cis_set_error(CIS_ERR_BAD_ARG, "cis_resize_concat_bf16: slices must be 8-channel aligned");
    total += srcs[i].chunks;
  }
  if ((dp | dc) & 7) return cis_set_error(CIS_ERR_BAD_ARG, "cis_resize_concat_bf16: destination must be 8-channel aligned");
  if ((size_t)N * OH > 65535 || (size_t)OW * total > 0x7fffffff) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_resize_concat_bf16: too many rows");
  if (OH == 2 * H && OW == 2 * W) {
    CIS_LAUNCH(resize_concat_x2_bf16_kernel, dim3((unsigned)((W * total + 255) / 256), (unsigned)(N * H)), 256, 0, ST, a, N, H, W, (mbf)dst, dp, dc, total);
    return cis_check_launch("resize_concat_x2_bf16");
  }
  CIS_LAUNCH(resize_concat_bf16_kernel, dim3((unsigned)((OW * total + 255) / 256), (unsigned)(N * OH)), 256, 0, ST, a, N, H, W, (mbf)dst, dp, dc, OH, OW,
             total);
  return cis_check_launch("resize_concat_bf16");
}
int cis_resize_concat_bf16_bwd(const void* ddst, int32_t dp, int32_t dc, int32_t N, int32_t OH, int32_t OW, const CisSrc* grads, const int32_t* want,
                               const int32_t* accumulate, int32_t nsrc, int32_t H, int32_t W, cis_stream_t stream) {
  if (!grads || nsrc < 1 || nsrc > CIS_MAX_SRC) return cis_set_error(CIS_ERR_BAD_ARG, "cis_resize_concat_bf16_bwd: 1..4 sources");
  RcGradArgs a;
  a.nsrc = nsrc;
  int total = 0;
  for (int i = 0; i < nsrc; ++i) {
    a.s[i].ptr = const_cast<void*>(grads[i].ptr);
    a.s[i].pitch = grads[i].pitch;
    a.s[i].c_off = grads[i].c_off;
    a.s[i].chunks = grads[i].chunks;
    a.s[i].n_mod = grads[i].n_mod;
    a.s[i].want = want[i];
    a.s[i].accumulate = accumulate[i];
    if (want[i] && (!grads[i].ptr || ((grads[i].pitch | grads[i].c_off) & 7))) return cis_set_error(CIS_ERR_BAD_ARG, "cis_resize_concat_bf16_bwd: bad gradient slice");
    if (grads[i].n_mod && N % grads[i].n_mod) return cis_set_error(CIS_ERR_BAD_ARG, "cis_resize_concat_bf16_bwd: N must be a multiple of n_mod");
    total += grads[i].chunks;
  }
  if ((size_t)N * H > 65535 || (size_t)W * total > 0x7fffffff) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_resize_concat_bf16_bwd: too many rows");
  CIS_LAUNCH(resize_concat_bf16_bwd_kernel, dim3((unsigned)((W * total + 255) / 256), (unsigned)(N * H)), 256, 0, ST, (cbf)ddst, dp, dc, N, OH, OW, a, H,
             W, total);
  return cis_check_launch("resize_concat_bf16_bwd");
}
int cis_resize_bilinear_f32(const float* src, int32_t N, int32_t H, int32_t W, int32_t C, float* dst, int32_t OH, int32_t OW, float scale,
                            cis_stream_t stream) {
  CIS_LAUNCH(resize_bilinear_f32_kernel, nblk((size_t)N * OH * OW), 256, 0, ST, src, N, H, W, C, dst, OH, OW, scale);
  return cis_check_launch("resize_bilinear_f32");
}
int cis_crop_resize_bilinear_f32(const float* src, int32_t Hs, int32_t Ws, int32_t C, int32_t y0, int32_t x0, int32_t ch, int32_t cw, float* dst,
                                 int32_t OH, int32_t OW, cis_stream_t stream) {
  if (!src || !dst || y0 < 0 || x0 < 0 || ch < 1 || cw < 1 || y0 + ch > Hs || x0 + cw > Ws || OH < 1 || OW < 1)
    return cis_set_error(CIS_ERR_BAD_ARG, "cis_crop_resize_bilinear_f32: crop box outside the image");
  CIS_LAUNCH(crop_resize_f32_kernel, nblk((size_t)OH * OW), 256, 0, ST, src, Ws, C, y0, x0, ch, cw, dst, OH, OW);
  return cis_check_launch("crop_resize_f32");
}
int cis_upsample_nn2x(const void* src, int32_t N, int32_t H, int32_t W, int32_t pitch, void* dst, cis_stream_t stream) {
  if ((size_t)N * 2 * H > 65535) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_upsample_nn2x: too many rows");
  CIS_LAUNCH(upsample_nn2x_kernel, dim3((unsigned)((2 * W * (pitch / 8) + 255) / 256), (unsigned)(N * 2 * H)), 256, 0, ST, (cbf)src, N, H, W, pitch,
             (mbf)dst);
  return cis_check_launch("upsample_nn2x");
}
int cis_upsample_nn2x_bwd(const void* dd, int32_t N, int32_t H, int32_t W, int32_t pitch, void* ds, int32_t accumulate, cis_stream_t stream) {
  if ((size_t)N * H > 65535) return cis_set_error(CIS_ERR_UNSUPPORTED, "cis_upsample_nn2x_bwd: too many rows");
  CIS_LAUNCH(upsample_nn2x_bwd_kernel, dim3((unsigned)((W * (pitch / 8) + 255) / 256), (unsigned)(N * H)), 256, 0, ST, (cbf)dd, N, H, W, pitch, (mbf)ds,
             accumulate);
  return cis_check_launch("upsample_nn2x_bwd");
}
int cis_resize_nn_f32(const float* src, int32_t N, int32_t H, int32_t W, int32_t C, float* dst, int32_t OH, int32_t OW, cis_stream_t stream) {
  CIS_LAUNCH(resize_nn_f32_kernel, nblk((size_t)N * OH * OW), 256, 0, ST, src, N, H, W, C, dst, OH, OW);
  return cis_check_launch("resize_nn_f32");
}
int cis_warp_costvol(const void* c1, int32_t c1p, int32_t c1o, const void* c2, int32_t c2p, int32_t c2o, const float* flow, float fs, int32_t B,
                     int32_t h, int32_t w, int32_t C, void* out, int32_t op, int32_t oo, cis_stream_t stream) {
  if (h < 2 || w < 2) return cis_set_error(CIS_ERR_BAD_ARG, "cis_warp_costvol: needs h,w >= 2 (core_warp.py:188)");
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(warp_costvol_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCvSmem);
    if (e != cudaSuccess) return cis_set_cuda_error(e, "cudaFuncSetAttribute(warp_costvol)");
    attr = true;
  }
  dim3 grid((w + kCvTW - 1) / kCvTW, (h + kCvTH - 1) / kCvTH, B);
  CIS_LAUNCH(warp_costvol_kernel, grid, 256, kCvSmem, ST, (cbf)c1, c1p, c1o, (cbf)c2, c2p, c2o, flow, fs, B, h, w, C, (mbf)out, op, oo);
  return cis_check_launch("warp_costvol");
}
int cis_dense_image_warp(const void* img, int32_t pitch, int32_t coff, const float* flow, float fs, int32_t B, int32_t h, int32_t w, int32_t C,
                         void* out, int32_t op, cis_stream_t stream) {
  const int chunks = (C + 7) / 8;
  CIS_LAUNCH(dense_image_warp_kernel, nblk((size_t)B * h * w * chunks), 256, 0, ST, (cbf)img, pitch, coff, flow, fs, B, h, w, chunks, (mbf)out, op);
  return cis_check_launch("dense_image_warp");
}
int cis_pack_f32_to_bf16(const float* src, int64_t npix, int32_t C, float offset, void* dst, int32_t dp, int32_t dc, cis_stream_t stream) {
  if (C > 8) return cis_set_error(CIS_ERR_BAD_ARG, "cis_pack_f32_to_bf16: C > 8");
  CIS_LAUNCH(pack_f32_to_bf16_kernel, nblk((size_t)npix), 256, 0, ST, src, (size_t)npix, C, offset, (mbf)dst, dp, dc);
  return cis_check_launch("pack_f32_to_bf16");
}
int cis_flow_stats(const float* flow, int32_t B, int64_t hw, double* stats, cis_stream_t stream) {
  dim3 grid(64, B);
  CIS_LAUNCH(flow_stats_kernel, grid, 256, 0, ST, flow, (size_t)hw, stats);
  return cis_check_launch("flow_stats");
}
int cis_pack_generator_input(const float* image, const float* flow, const double* stats, int32_t B, int64_t hw, void* dst, cis_stream_t stream) {
  dim3 grid(nblk((size_t)hw), B);
  CIS_LAUNCH(pack_generator_input_kernel, grid, 256, 0, ST, image, flow, stats, (size_t)hw, (mbf)dst);
  return cis_check_launch("pack_generator_input");
}
int cis_mask_apply(const float* flow, const float* mask, int32_t B, int64_t hw, void* dst, cis_stream_t stream) {
  CIS_LAUNCH(mask_apply_kernel, nblk((size_t)B * hw), 256, 0, ST, flow, mask, (size_t)B * hw, (mbf)dst);
  return cis_check_launch("mask_apply");
}
int cis_charbonnier_sum(const float* gt, const float* pred, const float* mask, int32_t B, int64_t hw, int32_t C, int32_t mask_c, float cbn,
                        double* sums, cis_stream_t stream) {
  if (C < 1 || (mask_c != 1 && mask_c != C)) return cis_set_error(CIS_ERR_BAD_ARG, "cis_charbonnier_sum: mask must have 1 or C channels");
  dim3 grid(64, B);
  CIS_LAUNCH(charbonnier_sum_kernel, grid, 256, 0, ST, gt, pred, mask, (size_t)hw, C, mask_c, cbn, sums);
  return cis_check_launch("charbonnier_sum");
}
int cis_cis_loss_fwd(const float* flow, const float* mask, const float* flow1, int32_t B, int32_t H, int32_t W, int32_t h1, int32_t w1, float cbn,
                     double* sums, float* pred_out, cis_stream_t stream) {
  dim3 grid(148, B);
  CIS_LAUNCH(cis_loss_fwd_kernel, grid, 256, 0, ST, flow, mask, flow1, B, H, W, h1, w1, cbn, sums, pred_out);
  return cis_check_launch("cis_loss_fwd");
}
int cis_cis_loss_reduce(const double* sums, int32_t B, int32_t global_batch, int64_t hw, float epsilon, float* scalars, float* coef,
                        cis_stream_t stream) {
  CIS_LAUNCH(cis_loss_reduce_kernel, 1, 32, 0, ST, sums, B, global_batch, (double)hw, epsilon, scalars, coef);
  return cis_check_launch("cis_loss_reduce");
}
int cis_cis_loss_bwd(const float* flow, const float* mask, const float* flow1, const float* coef, const float* scalars, int32_t B, int32_t H,
                     int32_t W, int32_t h1, int32_t w1, float cbn, int32_t which, float* dpred, float* dmask, cis_stream_t stream) {
  dim3 grid(nblk((size_t)H * W), B);
  CIS_LAUNCH(cis_loss_bwd_kernel, grid, 256, 0, ST, flow, mask, flow1, coef, scalars, B, H, W, h1, w1, cbn, which, dpred, dmask);
  return cis_check_launch("cis_loss_bwd");
}
int cis_resize_f32_bwd_to_bf16(const float* dd, int32_t N, int32_t OH, int32_t OW, int32_t C, int32_t H, int32_t W, void* ds, int32_t sp,
                               cis_stream_t stream) {
  if (C > 8) return cis_set_error(CIS_ERR_BAD_ARG, "cis_resize_f32_bwd_to_bf16: C > 8");
  CIS_LAUNCH(resize_f32_bwd_to_bf16_kernel, nblk((size_t)N * H * W), 256, 0, ST, dd, N, OH, OW, C, H, W, (mbf)ds, sp);
  return cis_check_launch("resize_f32_bwd_to_bf16");
}
int cis_mask_bwd(const float* flow, const float* mask, const float* dmd, const void* din, int32_t B, int64_t hw, void* dlogits, cis_stream_t stream) {
  CIS_LAUNCH(mask_bwd_kernel, nblk((size_t)B * hw), 256, 0, ST, flow, mask, dmd, (cbf)din, (size_t)B * hw, (mbf)dlogits);
  return cis_check_launch("mask_bwd");
}
int cis_abs_sum(const float* g, int64_t n, float* stat, cis_stream_t stream) {
  CIS_LAUNCH(abs_sum_kernel, 296, 256, 0, ST, g, (size_t)n, stat);
  return cis_check_launch("abs_sum");
}
int cis_grad_avg_abs(const float* g, const int64_t* seg_off, int32_t nseg, float* out_avg, cis_stream_t stream) {
  CIS_LAUNCH(grad_avg_abs_kernel, dim3((unsigned)nseg, 16), 256, 0, ST, g, (const long long*)seg_off, nseg, out_avg);
  return cis_check_launch("grad_avg_abs");
}
int cis_clip_adam(float* param, float* m, float* v, const float* grad, int64_t n, float grad_scale, float clip, float lr, float beta1, float beta2,
                  float eps, int64_t* step_state, const float* avg_abs, int32_t can_change, uint64_t seed, cis_stream_t stream) {
  if (can_change && !avg_abs) return cis_set_error(CIS_ERR_BAD_ARG, "cis_clip_adam: can_change needs avg_abs");
  CIS_LAUNCH(clip_adam_kernel, nblk((size_t)n), 256, 0, ST, param, m, v, grad, (size_t)n, grad_scale, clip, lr, beta1, beta2, eps,
                                                    (const long long*)step_state, avg_abs, can_change, (unsigned long long)seed);
  CIS_LAUNCH(step_inc_kernel, 1, 1, 0, ST, (long long*)step_state);
  return cis_check_launch("clip_adam");
}
int cis_cast_f32_to_bf16(const float* src, int64_t n, void* dst, cis_stream_t stream) {
  CIS_LAUNCH(cast_f32_bf16_kernel, nblk((size_t)n), 256, 0, ST, src, (size_t)n, (mbf)dst);
  return cis_check_launch("cast_f32_to_bf16");
}
int cis_cast_bf16_to_f32(const void* src, int64_t npix, int32_t pitch, int32_t coff, int32_t C, float* dst, cis_stream_t stream) {
  CIS_LAUNCH(cast_bf16_f32_kernel, nblk((size_t)npix * C), 256, 0, ST, (cbf)src, (size_t)npix, pitch, coff, C, dst);
  return cis_check_launch("cast_bf16_to_f32");
}

}  // extern "C"
