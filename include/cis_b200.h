/* cis_b200.h - C ABI of libcis_b200.so: the sm_100a kernels behind the adversarial motion-segmentation hot path.
 *
 * The reference (antonilo/unsupervised_detection @ 46cae6e) has no FFI layer: its "operators" are TensorFlow 1.13 graph
 * ops called from Python (SURVEY.md section 8b).  Each entry point below replaces the TF op class used at the cited
 * reference call site.  All pointers are DEVICE pointers owned by the caller (torch-allocated), every call only enqueues
 * work on `stream` and returns immediately; return value 0 = OK, non-zero = CIS_ERR_* (see cis_last_error()).
 * No torch types appear in any signature.  Layout everywhere: NHWC, activations bf16 with the channel pitch a multiple
 * of 8 (16-byte pixels chunks), flows/masks/losses fp32.
 */
#ifndef CIS_B200_H_
#define CIS_B200_H_
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* cis_stream_t; /* cudaStream_t */

enum { CIS_OK = 0, CIS_ERR_BAD_ARG = 1, CIS_ERR_UNSUPPORTED = 2, CIS_ERR_CUDA = 3 };
enum { CIS_ACT_NONE = 0, CIS_ACT_ELU = 1, CIS_ACT_LEAKY = 2 };
enum { CIS_MAX_TAPS = 49, CIS_MAX_SRC = 4 };

/* One channel slice of a bf16 NHWC tensor: a member of a virtual concat (tf.concat, nets.py:78-105,
 * model_pwcnet.py:482-502) that is never materialised. */
typedef struct {
  const void* ptr; /* bf16 base of the underlying buffer [N,H,W,pitch] */
  int32_t pitch;   /* channels per pixel of the underlying buffer (multiple of 8) */
  int32_t c_off;   /* first channel of the slice (multiple of 8) */
  int32_t chunks;  /* slice width in 8-channel chunks */
  int32_t n_mod;   /* >0: batch index taken modulo n_mod (features shared by the 3 recover_net calls) */
} CisSrc;

/* Implicit-GEMM convolution on tcgen05 tensor cores: D[rows=(n,oh,ow)][BN] = sum_k A[row][k] * Wp[n][k],
 * A[row][(t,c)] = src[n, oh*sh + dh[t], ow*sw + dw[t], c] (zero outside the image = TF 'SAME' padding).
 * With suitable tap tables this one kernel is: tf.layers.conv2d / tf.nn.conv2d forward (convolution_utils.py:46,81;
 * model_pwcnet.py:161-165,484-504,562-574), its data gradient (stride 1: flipped taps; stride 2: four parity launches),
 * and tf.layers.conv2d_transpose k4 s2 (model_pwcnet.py:286; four parity launches). */
typedef struct {
  int32_t N, H, W;   /* source batch / height / width */
  int32_t OH, OW;    /* GEMM row grid; rows = N*OH*OW */
  int32_t sh, sw;    /* source coordinate = row coordinate * s + tap offset */
  int32_t ntaps;
  int16_t dh[CIS_MAX_TAPS];
  int16_t dw[CIS_MAX_TAPS];
  int32_t nsrc;
  CisSrc src[CIS_MAX_SRC];
  const void* wpack; /* halo=0: bf16 [n_tiles*BN][K_pad], K order (tap, concat channel), K_pad multiple of 64;
                        halo=1: pre-swizzled tiles from cis_pack_weights_tiled */
  int32_t K_pad;
  int32_t BN;        /* N tile: 16, 32, 64 or 128 */
  int32_t n_tiles;   /* grid.y; padded output channels = n_tiles*BN */
  const float* bias; /* fp32 [n_tiles*BN] or NULL */
  int32_t act;       /* CIS_ACT_* */
  float alpha;       /* leaky slope */
  int32_t DH, DW;    /* destination height / width */
  int32_t osh, osw, oa, ob; /* destination pixel = (oh*osh + oa, ow*osw + ob) */
  void* out;         /* bf16 destination or NULL */
  int32_t out_pitch, out_coff, out_ch;
  float* outf;       /* fp32 destination or NULL */
  int32_t outf_pitch, outf_coff, outf_ch;
  const void* add_pre; /* bf16, added before the activation (gradient accumulation) */
  int32_t add_pre_pitch, add_pre_coff;
  const float* addf_pre; /* fp32, added before the activation (PWC flow + context residual, model_pwcnet.py:576) */
  int32_t addf_pitch, addf_coff;
  const void* add_post; /* bf16, added after the activation (generator skips, nets.py:29,32,33) */
  int32_t add_post_pitch, add_post_coff;
  int32_t mode;      /* 0 normal; 1: outf[pix] = sigmoid((l0 - l1)/10)  (nets.py:38-41) */
  /* halo-resident variant (stride-1 gathers only): the CTA tile is MT stacked 16x8-pixel blocks of dilation phase (a,b);
   * the (16*MT+ey) x (8+ex) input halo of a 64-channel chunk is staged ONCE in shared memory and all taps read it through
   * shifted UMMA descriptors.  dh/dw then hold tap offsets >= 0 relative to the halo origin, in units of `dil` pixels. */
  int32_t halo;      /* 0: generic per-tap gather kernel, 1: halo-resident kernel */
  int32_t dil;       /* dilation = phase period (1 for undilated) */
  int32_t MT;        /* 1..4 stacked M tiles (MT*BN <= 512 TMEM columns) */
  int32_t hoy, hox;  /* halo origin relative to the tile origin (phase units, <= 0) */
  int32_t ey, ex;    /* halo extent beyond the tile (max tap offset) */
  /* Split-K for launches that cover only a few SMs (low-resolution layers): grid.z = splits CTAs share one output tile, each reduces a
   * range of the K loop (64-wide K blocks for the gather kernel, 64-channel chunks for the halo kernel) and stores its partial fp32
   * tile to a private slice of sk_scratch; a second kernel launched by the same call sums the slices in a fixed order
   * (deterministic) and runs the fused epilogue spread over many CTAs. */
  int32_t splits;        /* 0/1 = off */
  float* sk_scratch;     /* >= tiles * splits * 128 * BN floats (tiles = grid.x * grid.y * MT); need not be initialised */
  int32_t* sk_counters;  /* must be NULL (the single-launch ticket mode of round 1 was removed; the field keeps the struct layout) */
  /* Stride-2 forward convolution on the halo kernel (halo = 1, sh = sw = 1 in this descriptor, H x W = the INPUT size): the input is
   * read as nph = 4 space-to-depth phases in(2y + py, 2x + px), phase index py*2 + px; taps are listed phase by phase in PHASE
   * coordinates (dh/dw relative to the halo origin of the phase images) and taps [ph_tap[i], ph_tap[i+1]) belong to phase i.
   * nph = 0/1: ordinary stride-1 gather. */
  int32_t nph;
  int32_t ph_tap[5];
  /* 1: the `splits` CTAs of a tile form a thread-block cluster (2..8 CTAs) and reduce their partial accumulators through distributed
   * shared memory inside the conv kernel (fixed summation order, fused epilogue spread over the cluster): no sk_scratch, no second launch. */
  int32_t sk_cluster;
  /* Grouped launch (halo kernel, splits <= 1): nsub = 2..4 sub-problems that share sources, epilogue, BN / n_tiles / MT and the halo box
   * (ey, ex) but have their own tap set, halo origin, packed weights, output extent and output offset -- the four output-parity
   * launches of a stride-2 data gradient or of conv2d_transpose(k4, s2) as ONE launch (blockIdx.z = sub-problem).  The taps of all
   * sub-problems are listed back to back in dh / dw (ntaps = their total); nsub = 0/1: ordinary launch. */
  int32_t nsub;
  struct {
    int32_t tap0, ntaps;      /* this sub-problem's taps: dh/dw[tap0 .. tap0 + ntaps) */
    int32_t hoy, hox;         /* halo origin relative to the output tile */
    int32_t OH, OW, oa, ob;   /* output extent and offset inside the (DH, DW) destination grid (stride osh / osw) */
    const void* wpack;        /* pre-tiled weights of this sub-problem */
  } sub[4];
  /* Compact thin halo (halo = 1, all sources together <= 16 channels): the halo is staged as 8-channel planes of 16 B per pixel
   * ([plane][Hh][Wh][8], SWIZZLE_NONE) and every "tap" of dh / dw / ntaps / ph_tap / sub[] is one K=16 MMA: for 8-channel inputs two
   * x-adjacent taps (the second K half is the next pixel), for 16 channels one tap (the second K half is the next plane).  wpack then
   * holds one BN x 32 B no-swizzle tile per MMA (cis_pack_weights_tiled, layout 1). */
  int32_t thin;
} CisConv;

/* Weight gradient of the same convolution: dWp[co][(t,c)] = sum_rows g[row][co] * A[row][(t,c)]  (fp32).  The reduction over rows
 * is split over `splits` CTAs per column tile; every split writes its own private slice of Cout x K_pad floats with plain stores
 * (element order: [co][K_pad] for tma == 2, float4 columns [K_pad/4][co][4] for tma 0 / 1 -- see cis_unpack_wgrad's `layout`)
 * (no atomics, nothing to zero) and cis_unpack_wgrad sums the slices in a fixed order -- the weight gradient is bit-reproducible.
 * Replaces the conv2d backprop-filter ops TF1 emits for tf.gradients (loss_utils.py:17). */
typedef struct {
  int32_t N, H, W, OH, OW, sh, sw, ntaps;
  int16_t dh[CIS_MAX_TAPS];
  int16_t dw[CIS_MAX_TAPS];
  int32_t nsrc;
  CisSrc src[CIS_MAX_SRC];
  const void* g;     /* bf16 gradient w.r.t. the pre-activation output on the (n,oh,ow) row grid */
  int32_t g_pitch, g_coff, g_chunks;
  float* dwp;        /* fp32 [splits][Cout][K_pad] private slices; every split must own >= 1 reduction block (ceil-division on the host) */
  int32_t Cout;      /* <= 128 */
  int32_t K_pad;
  int32_t splits;    /* split-K factor (grid.y) */
  int32_t tma;       /* 2: experimental halo-resident variant of 1 (same dwp layout; one activation halo per pixel tile, taps read in place);
                        1: stride-1 layer, operands fetched as 8x8-pixel TMA tiles; dwp columns are then laid out per tap in
                        64-channel groups: col = (tap*ceil(Cin8/64) + chunk64)*64 + c, K_pad = that extent rounded to 128 */
} CisWgrad;

const char* cis_last_error(void);
int cis_version(void);
/* Host-side CRC-32C (Castagnoli, reflected 0x82F63B78), extend form: returns crc32c(concat(A, data)) given crc = crc32c(A)
 * (pass 0 to start).  Used by the TF tensor-bundle checkpoint reader/writer (SURVEY 8f-1); it replaces
 * tensorflow/core/lib/hash/crc32c.h (TensorFlow 1.13, third-party, not vendored in the reference) behind
 * tf.train.Saver (models/adversarial_learner.py:326-331).  Not a stream operation; no GPU needed. */
uint32_t cis_crc32c(uint32_t crc, const void* data, size_t n);
/* Host-side frame preprocessing for the dataset readers (no GPU, not stream operations; thread-safe, callers run them from a thread pool).
 * tf.image.resize_images legacy bilinear on an HWC float image, and the fused decode-side step of preprocess_image
 * (data/davis2016_data_utils.py:84-90 of the reference): BGR uint8 -> RGB float v/255-0.5 -> legacy bilinear to OH x OW. */
int cis_host_resize_bilinear_legacy(const float* src, int32_t H, int32_t W, int32_t C, float* dst, int32_t OH, int32_t OW);
int cis_host_bgr8_to_rgb_resized(const unsigned char* bgr, int32_t H, int32_t W, float* dst, int32_t OH, int32_t OW);

int cis_conv_igemm(const CisConv* d, cis_stream_t stream);
/* which launches use the persistent warp-specialised halo kernel: 0 none, 1 thin single-chunk layers (default), 2 all eligible,
 * 3 = 1 + the weight-stationary variant for thin layers whose whole weight set fits in shared memory (experimental),
 * -1 back to the default / CIS_PERSIST_MODE environment variable.  Host-side switch, not a stream operation. */
int cis_set_persist_mode(int mode);
int cis_conv_wgrad(const CisWgrad* d, cis_stream_t stream);

/* ---- parameter-space helpers (fp32 master weights <-> packed bf16 operands) ---- */
/* wp[n][k] = (kmap[k] >= 0 && ne >= 0) ? w[kmap[k] + ne*sn] : 0 for n < rows, ne = nmap ? nmap[n] : (n < cout ? n : -1). */
int cis_pack_weights(const float* w, const int32_t* kmap, int32_t K_pad, int32_t rows, int32_t cout, int32_t sn, const int32_t* nmap,
                     void* wp, cis_stream_t stream);
/* halo-kernel operand: out[(ny, chunk, tap)][n][64] bf16 blocks of BN x 128 B with the SWIZZLE_128B pattern pre-applied; kmap is the
 * same tap-major map (k = tap*cin8 + channel).  layout 1 (compact thin halo, CisConv.thin): cin8 = 16, one BN x 32 B no-swizzle
 * block [K half][n][8] per MMA ("tap"). */
int cis_pack_weights_tiled(const float* w, const int32_t* kmap, int32_t cin8, int32_t ntaps, int32_t n_tiles, int32_t BN, int32_t cout,
                           int32_t sn, const int32_t* nmap, void* out, int32_t layout, cis_stream_t stream);
/* dw[kmap[k] + n] = sum_{s < nsplit} dwp[s](n, k) for kmap[k] >= 0, n < cout (fixed summation order; forward orientation, sn = 1);
 * and, when colpart != NULL, the bias gradient db[c] = sum_{b < nblocks} colpart[b][c], c < nch (the partials of cis_colsum).
 * layout = how cis_conv_wgrad stored a slice: 0 = [cout][K_pad] (CisWgrad.tma == 2), 1 = float4 columns [K_pad/4][cout][4] (tma 0 / 1). */
int cis_unpack_wgrad(const float* dwp, const int32_t* kmap, int32_t K_pad, int32_t cout, int32_t nsplit, float* dw, const float* colpart,
                     int32_t nblocks, int32_t nch, float* db, int32_t layout, cis_stream_t stream);
/* tf.layers.batch_normalization in inference mode folded into the conv (convolution_utils.py:46-51):
 * w_eff = w * gamma/sqrt(1+1e-3); b_eff = bias*gamma/sqrt(1+1e-3) + beta. */
int cis_bn_fold(const float* w, const float* bias, const float* gamma, const float* beta, int64_t nw, int32_t cout, float* w_eff,
                float* b_eff, cis_stream_t stream);
/* chain rule back to (w, bias, gamma, beta) from (dw_eff, db_eff); dw_eff is overwritten in place by dw. */
int cis_bn_chain(const float* w, const float* bias, const float* gamma, float* dw_eff_to_dw, const float* db_eff, int64_t nw,
                 int32_t cout, float* dbias, float* dgamma, float* dbeta, cis_stream_t stream);

/* Multi-job form of the five parameter-space ops above: ONE launch over a flat grid of 256-thread blocks.  A job holds the arguments of
 * the single-launch entry point of its kind in order: pointers in p[], the size_t argument (nw) in n, the int arguments in i[0..6]
 * (bn_chain: p[0..7] = w, bias, gamma, dw_eff, db_eff, dbias, dgamma, dbeta), and in i[7] the index of its first block; job j owns blocks
 * [i[7] of j, i[7] of j+1) and needs ceil(elements / 256) of them (bn_chain: cout).  The table lives in device memory, sorted by i[7];
 * total_blocks = the sum.  Jobs of one launch must not depend on each other. */
enum { CIS_JOB_PACK = 0, CIS_JOB_PACK_TILED = 1, CIS_JOB_UNPACK = 2, CIS_JOB_BN_FOLD = 3, CIS_JOB_BN_CHAIN = 4 };
typedef struct {
  int32_t kind;
  int32_t i[8];
  int64_t n;
  const void* p[8];
} CisParamJob;
int cis_param_multi(const CisParamJob* jobs_dev, int32_t njobs, int32_t total_blocks, cis_stream_t stream);

/* ---- elementwise / reduction helpers on bf16 NHWC slices ---- */
/* g *= act'(y - res)   (ELU: u>0 ? 1 : u+1; leaky: u>0 ? 1 : alpha) */
int cis_dact_mul(void* g, int32_t g_pitch, int32_t g_coff, const void* y, int32_t y_pitch, int32_t y_coff, const void* res,
                 int32_t res_pitch, int32_t res_coff, int64_t npix, int32_t chunks, int32_t act, float alpha, cis_stream_t stream);
/* dst (=|+=) sum_{j<reps} src[(pix + j*npix_dst)]  : gradient accumulation and the 3-call fold of shared features */
int cis_add_slice(void* dst, int32_t dst_pitch, int32_t dst_coff, const void* src, int32_t src_pitch, int32_t src_coff,
                  int64_t npix_dst, int32_t chunks, int32_t reps, int32_t accumulate, cis_stream_t stream);
/* part[b][c] = sum over the pixels of block b of g[pix][c], c < nch, b < nblocks (<= 592): per-block partial column sums, no atomics;
 * cis_unpack_wgrad adds them up in block order (deterministic bias gradient). */
int cis_colsum(const void* g, int32_t g_pitch, int32_t g_coff, int64_t npix, int32_t nch, float* part, int32_t nblocks, cis_stream_t stream);

/* zero-fill of the small accumulators a step starts from (flow statistics, loss sums, gradient magnitude): stream-ordered memset */
int cis_zero(void* ptr, int64_t nbytes, cis_stream_t stream);

/* cis_dact_mul and cis_colsum of the same gradient slice in one pass: g *= act'(y - res) in place, part[b][c] = block b's column sums of
 * the rounded product (bit-identical to the two separate calls with the same nblocks). */
int cis_dact_colsum(void* g, int32_t g_pitch, int32_t g_coff, const void* y, int32_t y_pitch, int32_t y_coff, const void* res,
                    int32_t res_pitch, int32_t res_coff, int64_t npix, int32_t nch, int32_t act, float alpha, float* part, int32_t nblocks,
                    cis_stream_t stream);

/* ---- resampling (App. A.5/A.6 semantics) ---- */
/* tf.image.resize_images / resize_bilinear legacy (convolution_utils.py:88, nets.py:108) on a bf16 slice */
int cis_resize_bilinear_bf16(const void* src, int32_t s_pitch, int32_t s_coff, int32_t N, int32_t H, int32_t W, void* dst,
                             int32_t d_pitch, int32_t d_coff, int32_t OH, int32_t OW, int32_t chunks, cis_stream_t stream);
/* fused resize + concat of the recover decoder (convolution_utils.py:87-90 feeding nets.py:80-105): up to 4 sources of one resolution
 * (channel slices, batch-broadcast when n_mod > 0) -> legacy-bilinear to OH x OW -> side by side into one destination slice.
 * H x W == OH x OW makes it a plain concat copy. */
int cis_resize_concat_bf16(const CisSrc* srcs, int32_t nsrc, int32_t N, int32_t H, int32_t W, void* dst, int32_t d_pitch, int32_t d_coff,
                           int32_t OH, int32_t OW, cis_stream_t stream);
/* its transpose: for every source i with want[i]: grads[i] (=|+= when accumulate[i]) sum over broadcast replicas of R^T ddst[slice i];
 * grads[i].chunks must equal the forward source's (it positions the slice inside ddst), N = batch rows of ddst processed. */
int cis_resize_concat_bf16_bwd(const void* ddst, int32_t d_pitch, int32_t d_coff, int32_t N, int32_t OH, int32_t OW, const CisSrc* grads,
                               const int32_t* want, const int32_t* accumulate, int32_t nsrc, int32_t H, int32_t W, cis_stream_t stream);
/* its transpose: dsrc (=|+=) R^T ddst */
int cis_resize_bilinear_bf16_bwd(const void* ddst, int32_t d_pitch, int32_t d_coff, int32_t N, int32_t OH, int32_t OW, void* dsrc,
                                 int32_t s_pitch, int32_t s_coff, int32_t H, int32_t W, int32_t chunks, int32_t accumulate,
                                 cis_stream_t stream);
/* fp32, C channels: dst = scale * resize(src)  (adversarial_learner.py:87-97, model_pwcnet.py:646) */
int cis_resize_bilinear_f32(const float* src, int32_t N, int32_t H, int32_t W, int32_t C, float* dst, int32_t OH, int32_t OW,
                            float scale, cis_stream_t stream);
/* tf.image.resize_nearest_neighbor(align_corners=True) x2 (convolution_utils.py:71) and its transpose */
int cis_upsample_nn2x(const void* src, int32_t N, int32_t H, int32_t W, int32_t pitch, void* dst, cis_stream_t stream);
int cis_upsample_nn2x_bwd(const void* ddst, int32_t N, int32_t H, int32_t W, int32_t pitch, void* dsrc, int32_t accumulate,
                          cis_stream_t stream);
/* central crop (box y0, x0, ch, cw of ONE Hs x Ws x C fp32 NHWC image) resized back to OH x OW with the legacy bilinear rule: the
 * multi-crop test-time augmentation of test_generator_ensemble (data/davis2016_data_utils.py:130-134, 328-354) on the device */
int cis_crop_resize_bilinear_f32(const float* src, int32_t Hs, int32_t Ws, int32_t C, int32_t y0, int32_t x0, int32_t ch, int32_t cw, float* dst,
                                 int32_t OH, int32_t OW, cis_stream_t stream);
/* tf.image.resize_images(NEAREST_NEIGHBOR) for GT masks (adversarial_learner.py:92-94) */
int cis_resize_nn_f32(const float* src, int32_t N, int32_t H, int32_t W, int32_t C, float* dst, int32_t OH, int32_t OW,
                      cis_stream_t stream);

/* ---- PWC-Net warp + cost volume (core_warp.py:153-202 fused into core_costvol.py:20-40) ----
 * out[b,y,x,9*dy+dx] = leaky0.1( mean_c c1[b,y,x,c] * warp(c2, flow)[b,y+dy-4,x+dx-4,c] ), zero outside; flow may be
 * NULL (level 6: no warp).  flow is fp32 [B,h,w,2] and is multiplied by flow_scale (model_pwcnet.py:616-617). */
int cis_warp_costvol(const void* c1, int32_t c1_pitch, int32_t c1_coff, const void* c2, int32_t c2_pitch, int32_t c2_coff,
                     const float* flow, float flow_scale, int32_t B, int32_t h, int32_t w, int32_t C, void* out, int32_t out_pitch,
                     int32_t out_coff, cis_stream_t stream);
/* standalone dense_image_warp (core_warp.py:153) on a bf16 slice -> bf16, for parity tests of the gather */
int cis_dense_image_warp(const void* img, int32_t pitch, int32_t coff, const float* flow, float flow_scale, int32_t B, int32_t h,
                         int32_t w, int32_t C, void* out, int32_t out_pitch, cis_stream_t stream);

/* ---- input packing ---- */
/* bf16 [N,H,W,8] = (src fp32 [N,H,W,C] + offset), zero padded (model_pwcnet.py:39-56 adapt_x) */
int cis_pack_f32_to_bf16(const float* src, int64_t npix, int32_t C, float offset, void* dst, int32_t d_pitch, int32_t d_coff,
                         cis_stream_t stream);
/* per-sample sums for tf.nn.moments (flow_utils.py:10): stats[b] = {sum f0, sum f1, sum f0^2, sum f1^2} (double, zeroed) */
int cis_flow_stats(const float* flow, int32_t B, int64_t hw, double* stats, cis_stream_t stream);
/* generator input = concat(image, (flow-mean)/sqrt(var)) -> bf16 [B,H,W,8]  (nets.py:14, flow_utils.py:5-12) */
int cis_pack_generator_input(const float* image, const float* flow, const double* stats, int32_t B, int64_t hw, void* dst,
                             cis_stream_t stream);

/* ---- mask (x) flow + Charbonnier contextual-information loss (adversarial_learner.py:107-110,141-204) ---- */
/* recover inputs, batch 3B: [flow*(1-m),1,1-m | flow*m,1,m | 0,0,1,0] -> bf16 [3B,H,W,8] (nets.py:50-53) */
int cis_mask_apply(const float* flow, const float* mask, int32_t B, int64_t hw, void* dst, cis_stream_t stream);
/* stand-alone charbonnier_loss (loss_utils.py:34-51): sums[b] += sum over pixels and C channels of ((gt-pred)^2 + 1e-6)^cbn * mask;
 * mask_c = 1 (one value per pixel) or C (one per element); sums = double [B], zeroed by the caller */
int cis_charbonnier_sum(const float* gt, const float* pred, const float* mask, int32_t B, int64_t hw, int32_t C, int32_t mask_c, float cbn,
                        double* sums, cis_stream_t stream);
/* sums[b] = {rec, rec_c, prior, den, den_c} (fp32 via double atomics; zeroed).  flow1 = fp32 [3B,H/2,W/2,2] recover
 * outputs before the final bilinear x2 (nets.py:108), which is fused here. */
int cis_cis_loss_fwd(const float* flow, const float* mask, const float* flow1, int32_t B, int32_t H, int32_t W, int32_t h1,
                     int32_t w1, float cbn, double* sums, float* pred_out /* optional [3B,H,W,2] */, cis_stream_t stream);
/* scalars[0]=generator loss, [1]=recover loss, [2]=red_rate, [3]=red_rate_compl, [4]=1/(H*W*global_batch);
 * coef[b*4..] = per-sample partial derivatives of the generator loss w.r.t. {rec, den, rec_c, den_c}.
 * global_batch = config.batch_size of the whole (data-parallel) job; losses are this rank's partial sums / global_batch. */
int cis_cis_loss_reduce(const double* sums, int32_t B, int32_t global_batch, int64_t hw, float epsilon, float* scalars, float* coef,
                        cis_stream_t stream);
/* which = 0: d recover_loss, 1: d generator_loss.  Writes dpred [3B,H,W,2] fp32 and (generator) the direct dL/dmask term. */
int cis_cis_loss_bwd(const float* flow, const float* mask, const float* flow1, const float* coef, const float* scalars, int32_t B,
                     int32_t H, int32_t W, int32_t h1, int32_t w1, float cbn, int32_t which, float* dpred, float* dmask,
                     cis_stream_t stream);
/* transpose of the final x2 resize: dflow1 [3B,h1,w1,2] -> bf16 [3B,h1,w1,8] gradient for the flow1 conv */
int cis_resize_f32_bwd_to_bf16(const float* ddst, int32_t N, int32_t OH, int32_t OW, int32_t C, int32_t H, int32_t W, void* dsrc,
                               int32_t s_pitch, cis_stream_t stream);
/* mask backward: dmask += chain through the recover inputs (d_in bf16 [>=2B,H,W,8], gradient of cis_mask_apply's output);
 * then through softmax(x/10)[0] -> bf16 gradient of the 2 logits [B,H,W,8]. */
int cis_mask_bwd(const float* flow, const float* mask, const float* dmask_direct, const void* d_in, int32_t B, int64_t hw,
                 void* dlogits, cis_stream_t stream);

/* ---- optimiser: clip / noise + TF-Adam (loss_utils.py:12-32, adversarial_learner.py:216-217) ---- */
/* stat[0] += sum|g| over [0,n)  (zeroed by caller); used for the can_change test */
int cis_abs_sum(const float* g, int64_t n, float* stat, cis_stream_t stream);
/* out_avg += mean over variables of mean|g_v| (loss_utils.py:19-20); seg = int64 [nseg][2] = {start,end} of each variable */
int cis_grad_avg_abs(const float* g, const int64_t* seg_off, int32_t nseg, float* out_avg, cis_stream_t stream);
/* step_state: device int64 {t}; advanced by this call.  can_change != 0 enables the noise branch on *avg_abs < 1e-5. */
int cis_clip_adam(float* param, float* m, float* v, const float* grad, int64_t n, float grad_scale, float clip, float lr, float beta1,
                  float beta2, float eps, int64_t* step_state, const float* avg_abs, int32_t can_change, uint64_t seed,
                  cis_stream_t stream);
int cis_cast_f32_to_bf16(const float* src, int64_t n, void* dst, cis_stream_t stream);
int cis_cast_bf16_to_f32(const void* src, int64_t npix, int32_t pitch, int32_t coff, int32_t C, float* dst, cis_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CIS_B200_H_ */
