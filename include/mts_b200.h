/* mts_b200.h -- C ABI of libmts_b200.so: the B200 (sm_100a) hot path of the multimodal topic segmenter.
 *
 * The reference (Ighina/MultimodalTopicSegmentation) is pure Python: it has no FFI of its own.  The
 * boundary it offers for this path is the Python duck type that `TextSegmenter` calls on `self.model`
 * (models/lightning_model.py:293-305, 333-349, 587-594, 682).  Each entry point below replaces the
 * library call(s) that one reference line makes, so that the host-side mirror in
 * multimodaltopicsegmentation_b200/modules.py can keep the reference's signatures.  INTEGRATION.md shows
 * the ctypes binding a maintainer would add on the reference side.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`; tensors are dense row-major
 *     fp32 unless stated; `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - no allocation, no ownership transfer, no host synchronisation inside any call;
 *   - return value: 0 on success, a positive cudaError_t on a CUDA failure, a negative MTS_E_* code on a
 *     rejected argument.  Nothing falls back to the CPU.
 */
#ifndef MTS_B200_H_
#define MTS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MTS_E_BADARG (-1)    /* null pointer / non-positive size */
#define MTS_E_UNSUPPORTED (-2) /* shape outside what the kernels implement (message via mts_last_error) */
#define MTS_E_NODEVICE (-3)  /* no sm_100 device */

int mts_version(void);                 /* ABI version, bumped on any signature change */
const char *mts_last_error(void);      /* static string describing the last negative return on this thread */
int mts_device_ok(void);               /* 0 when the current device is compute capability 10.x */

/* ------------------------------------------------------------------------------------------------
 * Operand preparation.  The tensor-core GEMM (mts_gemm_tf32x3) takes every fp32 operand X [rows, K] as a pair
 *   hi : fp32 [rows, Kp]  the values themselves, zero beyond K (kind::tf32 reads the top 19 bits of each word)
 *   lo : the SAME byte size, holding bf16 [rows, 2 Kp]: per 16-wide K block 32 values, for an A operand
 *        [ bf16(x_k), k = 0..15 | bf16(x_k - trunc_tf32(x_k)), k = 0..15 ], for a B operand the halves swapped
 * with Kp = K rounded up to a multiple of 32.  Every kernel below that has (hi, lo) outputs writes this format
 * (A side unless it takes a `side` argument).
 * ---------------------------------------------------------------------------------------------- */

/* Early fusion (utils/load_datasets_precomputed.py:158-161 `torch.cat(embs, axis=-1)`) fused with the
 * time crop to max(lengths) and the hi/lo split:  out[b*T + t, :] = [src1[b,t,:D1] | src2[b,t,:D2] | 0-pad].
 * src batch strides are in elements (so a [B, T_in, D] tensor cropped to T <= T_in needs no copy);
 * src2 may be NULL (D2 = 0).  hi/lo: [B*T, Kp], Kp % 32 == 0, Kp >= D1 + D2. */
int mts_pack_rows_split(const float *src1, int64_t bstride1, int D1, const float *src2, int64_t bstride2, int D2,
                        int B, int T, int Kp, float *hi, float *lo, void *stream);

/* Generic 2-D split: src [rows, cols] (row stride `ld`) -> hi/lo [rows, Kp].  side: 0 = the matrix will be the A
 * operand of mts_gemm_tf32x3, 1 = the B operand (the two halves of the correction blocks are swapped, see below). */
int mts_split_tf32(const float *src, int64_t ld, int rows, int cols, int Kp, int side, float *hi, float *lo,
                   void *stream);

/* Transposed split for the weight-gradient GEMMs (a contraction over tokens needs both operands K-major along the
 * token axis):  out[c, r] = src[(r / T) * bstride + (r % T + shift) * ld + c] when 0 <= r % T + shift < lengths[r / T]
 * (lengths may be NULL: T), else 0;  hi/lo [cols, Kp], Kp % 32 == 0, Kp >= rows, columns >= rows zero.
 * shift in {-1, 0, +1}: the h_{t-1} / h_{t+1} operand of dW_hh without a shifted copy of the hidden states.
 * A plain [rows, cols] matrix: T = rows, bstride = 0. */
int mts_transpose_split(const float *src, int64_t bstride, int64_t ld, int rows, int cols, int T, int shift,
                        const int32_t *lengths, int Kp, int side, float *hi, float *lo, void *stream);

/* Device-side collater (the reference pads every batch on the host, EncoderDataset.py:91-152): episodes packed back
 * to back in src [sum(len), D] with offsets[E+1] (int64) and lengths[E] (int32); for the B episode ids of a batch
 *   out[b, t, :] = t < lengths[ids[b]] ? src[offsets[ids[b]] + t, :] : pad      (out [B,T,D]) */
int mts_gather_pad(const float *src, const int64_t *offsets, const int32_t *lengths, const int32_t *ids, int B, int T,
                   int D, float pad, float *out, void *stream);

/* Token rows between the padded layout [B*S, d] (to_padded = 0: src) and the ragged layout [sum(len), d]
 * (to_padded = 1: src), offsets int32 [B] = exclusive prefix sums of lengths.  to_padded = 1 fills the padded rows
 * with `pad`; to_padded = 0 copies the valid rows only.  d % 4 == 0.  See "Row layouts" below. */
int mts_ragged_copy(const float *src, float *dst, const int32_t *lengths, const int32_t *offsets, int B, int S, int d,
                    int to_padded, float pad, void *stream);

/* ------------------------------------------------------------------------------------------------
 * GEMM:  C[M,N] = A[M,K] * B[N,K]^T (+ bias[N]) (+ GELU), fp32 in / fp32 out.
 *   replaces: nn.LSTM's input projection (models/NeuralArchitectures.py:113), nn.Linear heads
 *   (models/CRF.py:299-310) and HF Longformer's dense layers (modeling_longformer.py:513-515,1067,1112,1126).
 * mts_gemm_tf32x3: tcgen05 + TMA, error-compensated TF32 (fp32-grade accuracy): hi(A) hi(B)^T on kind::tf32 plus
 *   the two 2^-11-sized correction terms as ONE bf16 product over the packed `lo` operands (the entry keeps its
 *   historical name; it issues 2, not 3, instruction streams per product).  A_hi/A_lo [M,Kp], B_hi/B_lo [N,Kp] as
 *   produced above (A side / B side); ldc in elements; epilogue: 0 none, 1 +bias, 2 +bias then GELU(erf).
 *   accumulate != 0 adds into C.  K is split automatically (few output tiles with long K; always beyond K = 3072:
 *   the tensor core truncates when aligning addends, a drift linear in K) and the partial tiles meet in C through
 *   fp32 atomics.
 * mts_gemm_f32: exact-fp32 CUDA-core GEMM, C[M,N] (+)= op(A) op(B), used for the gradient products whose
 *   reduction runs over sentences and to validate the tensor-core kernel.  layout 0: A[M,K] B[N,K]^T;
 *   2: A[M,K] B[K,N]; 3: A[K,M]^T B[K,N].  splits > 1 = split-K with atomics.  shift != 0 (layouts 2,3) reads
 *   B row k as row k+shift, zero unless 0 <= (k % T) + shift < lengths[k / T]: the h_{t-1}/h_{t+1} operand of
 *   dW_hh without a shifted copy of the hidden states. */
int mts_gemm_tf32x3(const float *A_hi, const float *A_lo, const float *B_hi, const float *B_lo, const float *bias,
                    float *C, int M, int N, int Kp, int64_t ldc, int epilogue, int accumulate, void *stream);
int mts_gemm_f32(const float *A, int64_t lda, const float *B, int64_t ldb, const float *bias, float *C, int64_t ldc,
                 int M, int N, int K, int layout, int epilogue, int accumulate, int splits, int shift, int T,
                 const int32_t *lengths, void *stream);
/* column sums out[n] (+)= sum_m X[m,n]  (bias gradients); ws >= mts_colsum_ws_bytes(M, N) bytes */
int64_t mts_colsum_ws_bytes(int M, int N);
int mts_colsum(const float *X, int64_t ld, int M, int N, float *out, int accumulate, void *ws, void *stream);

/* ------------------------------------------------------------------------------------------------
 * LSTM recurrence  (torch.nn.LSTM as called at models/NeuralArchitectures.py:39-43,113-115).
 * One call runs BOTH directions of one layer (and, for late fusion, of `n_enc` independent encoders
 * laid out back to back) over a batch of variable-length episodes.
 *
 *   gx      [n_enc, B*T, 2*4H]  input projection + (b_ih + b_hh); columns = [dir][gate i,f,g,o][unit]
 *   w_hh    [n_enc, 2, 4H, H]   recurrent weights (PyTorch layout, forward then reverse)
 *   lengths [B] int32           valid length per episode, 1 <= len <= T
 *   y       [B, T, n_enc*2H]    hidden states, zero at t >= len_b (pad_packed_sequence semantics);
 *                               columns = [enc][dir][unit]  (late fusion's torch.cat, models/CRF.py:425)
 *   gates   [n_enc, 2, B, T, 5, H] or NULL: i,f,g,o (post-activation) and c saved for the backward pass
 *   order   [B] int32 or NULL   episode ids sorted by decreasing length: tile i of the cluster kernel takes
 *                               order[8i .. 8i+7], so that the episodes of a tile finish together
 * H == 256 runs the persistent cluster kernel (W_hh resident in registers across 8 CTAs, h exchanged
 * through distributed shared memory); other H run a generic kernel. */
int mts_lstm_rec_fwd(const float *gx, const float *w_hh, const int32_t *lengths, const int32_t *order, int n_enc,
                     int B, int T, int H, float *y, float *gates, void *stream);

/* The same recurrence on the tensor cores (H == 256 only): W_hh kept on chip (tensor memory) for the whole sequence,
 * tiles of up to 16 episodes per 8-CTA cluster, tcgen05.mma per step, h exchanged through distributed shared memory.
 * Same arguments and results (to fp32 rounding) as mts_lstm_rec_fwd, plus y_corr [B*T, 2H] or NULL (n_enc == 1 only):
 * the packed bf16 correction operand of y (A side), so that the next layer's input projection reads (y, y_corr)
 * directly -- no split pass.  Two formulations exist: the default is the fp16-split kernel (mts_lstm_rec_fwd_h3 below,
 * 48 MMAs per step); MTS_REC_TC=tf32 in the environment selects mts_lstm_rec_fwd_tf32 (one TF32 product + one bf16
 * correction product, 64 MMAs per step, csrc/lstm_rec_tc.cu). */
int mts_lstm_rec_fwd_tc(const float *gx, const float *w_hh, const int32_t *lengths, const int32_t *order, int n_enc,
                        int B, int T, int H, float *y, float *gates, float *y_corr, void *stream);
int mts_lstm_rec_fwd_tf32(const float *gx, const float *w_hh, const int32_t *lengths, const int32_t *order, int n_enc,
                          int B, int T, int H, float *y, float *gates, float *y_corr, void *stream);

/* Early-fusion input projection without a concatenated copy (utils/load_datasets_precomputed.py:158-161 concatenates the
 * text and audio embeddings, NeuralArchitectures.py:113 projects them): C = [A1 | A2] B^T with the raw fp32 A operand
 * read in place from its one or two source matrices (A1 [M, D1] row stride ld1, A2 [M, D2] row stride ld2 or NULL) by the
 * TMA producer -- k-blocks below D1 / 32 from A1, the others from A2 -- and only the packed correction operand
 * A_lo [M, Kp], Kp = pad32(D1 + D2), prepared beforehand (mts_pack_rows_split with hi == NULL).  D1 % 32 == 0 when A2 is
 * given; row strides multiples of 4 floats.  Other arguments as mts_gemm_tf32x3. */
int mts_gemm_tf32x3_srcs(const float *A1, int D1, int64_t ld1, const float *A2, int D2, int64_t ld2, const float *A_lo,
                         const float *B_hi, const float *B_lo, const float *bias, float *C, int M, int N, int Kp, int64_t ldc,
                         int epilogue, int accumulate, void *stream);

/* Dense layer over FP16-SPLIT operands (HF LongformerSelfAttention q/k/v projections :514-516 and LongformerIntermediate
 * :1103-1116 in inference, where the A operand comes from a LayerNorm that knows its row): x = x1 + x2 with x1 = fp16(x s),
 * x2 = fp16(x s - x1), s an exact power-of-two scale per operand row.  C = (A1 B1^T + A2 B1^T + A1 B2^T) rs[m] cs[n] (+ bias,
 * epilogue 2: GELU): three kind::f16 tcgen05 products -- 6 instead of 8 MMAs per 32 k and half the operand bytes of
 * mts_gemm_tf32x3, relative error ~2^-22.  A_pieces [M][2][K] fp16 (mts_add_ln_fwd_f16 / mts_embed_ln_fwd_f16 write it),
 * B_pieces [N][2][K], row_scale [M] / col_scale [N] = 1 / s or NULL; K % 64 == 0, K <= 3072, M, N >= 256.  C_lo (optional):
 * the packed bf16 correction operand of C, for a following mts_gemm_tf32x3 (dense rows, N % 32 == 0). */
/* Early-fusion concat + crop (utils/load_datasets_precomputed.py:158-161, NeuralArchitectures.py:115) straight into the
 * fp16-split operand: pieces [B*T][2][K64] fp16 and row_scale [B*T] of the rows [src1[b, t, :] | src2[b, t, :]], t < T
 * (a warp owns a row: its maximum fixes the row's power-of-two scale).  D1, D2 % 4 == 0, D1 + D2 <= 2048, K64 % 64 == 0. */
int mts_pack_rows_f16(const float *src1, int64_t bstride1, int D1, const float *src2, int64_t bstride2, int D2, int B, int T,
                      int K64, void *pieces, float *row_scale, void *stream);
int mts_gemm_f16x3(const void *A_pieces, const void *B_pieces, const float *row_scale, const float *col_scale, const float *bias,
                   float *C, float *C_lo, int M, int N, int K, int64_t ldc, int epilogue, void *stream);

/* LongformerIntermediate (HF modeling_longformer.py:1103-1116: dense + GELU(erf)) when its output feeds the next dense
 * layer: C [M,N] = gelu(A B^T + bias) in fp32 -- which is its own `hi` operand -- and C_lo [M,N] = the packed correction
 * operand of C (A side), both written by the GEMM epilogue.  Replaces mts_gemm_tf32x3 + mts_gelu_split in inference
 * (training keeps the pre-activation).  N % 32 == 0, Kp % 32 == 0, Kp <= 3072, rows of C and C_lo dense (stride N). */
int mts_gemm_tf32x3_gelu_pair(const float *A_hi, const float *A_lo, const float *B_hi, const float *B_lo, const float *bias,
                              float *C, float *C_lo, int M, int N, int Kp, void *stream);

/* ---- bf16 path (explicit precision switch; fp32 stays the default and the parity contract) -----------------------
 * The same kernels with bf16 operands on kind::f16 MMAs only: per product one bf16 x bf16 term instead of the
 * error-compensated TF32 + bf16 pair.  State, gates, accumulation and every output stay fp32.  Tolerances per kernel
 * (measured against the fp32 oracle at T = 300 and T = 8192) are listed in DESIGN.md.
 *   mts_lstm_rec_fwd_tc_bf16 : nn.LSTM recurrence (NeuralArchitectures.py:113) with bf16(W_hh) bf16(h) products: 16 instead of
 *                              48 MMAs per step, half the h exchange.  Same arguments as mts_lstm_rec_fwd_tc.
 *   mts_gemm_bf16p           : C = A B^T (+ bias, epilogues as mts_gemm_tf32x3) from the PACKED operands alone: A_lo as every
 *                              producer writes it (side 0), B_lo = the weights packed with side 0 too.  The raw fp32 arrays
 *                              are not read: half the operand bytes, half the MMAs.
 *   mts_pack_rows_bf16in     : early-fusion concat + crop of BF16 embedding tensors (src1 [B,*,D1], src2 [B,*,D2], strides in
 *                              elements) straight into the packed operand: embeddings stored and shipped as bf16 halve the
 *                              host->device bytes of the path (utils/load_datasets_precomputed.py:158-161 is where the
 *                              reference concatenates fp32). */
int mts_lstm_rec_fwd_tc_bf16(const float *gx, const float *w_hh, const int32_t *lengths, const int32_t *order, int n_enc,
                             int B, int T, int H, float *y, float *gates, float *y_corr, void *stream);
int mts_gemm_bf16p(const float *A_lo, const float *B_lo, const float *bias, float *C, int M, int N, int Kp, int64_t ldc,
                   int epilogue, int accumulate, void *stream);
int mts_pack_rows_bf16in(const void *src1, int64_t bstride1, int D1, const void *src2, int64_t bstride2, int D2, int B, int T,
                         int Kp, float *lo, void *stream);
/* bf16 path of the windowed-attention encoder (inference; replaces, per layer, what HF LongformerLayer computes,
 * modeling_longformer.py:401-442, 481-639, 1060-1171, from models/RestrictedTransformerLayer.py:131):
 *   mts_gemm_bf16p_out16     : the q/k/v projection (LongformerSelfAttention.query/key/value, :503-505): mts_gemm_bf16p with
 *                              the bias epilogue, C stored as bf16 [M, ldc] = round-to-nearest-even of mts_gemm_bf16p's fp32
 *                              output.  N % 4 == 0, ldc % 4 == 0, Kp <= 3072 (no K split).
 *   mts_gemm_bf16p_gelu_pair : LongformerIntermediate (:1103-1116): the bf16-product twin of mts_gemm_tf32x3_gelu_pair,
 *                              C = gelu(A B^T + bias) fp32 [M, N] and its packed operand C_lo [M, N] (side 0).
 *   mts_embed_ln_fwd_bf16in  : LongformerEmbeddings (:401-442) = mts_embed_ln_fwd reading bf16 embeddings x; writes y fp32 and
 *                              its packed operand y_lo [rows, Kp] (Kp == d).
 *   mts_band_attn_fwd_bf16   : LongformerSelfAttention's banded softmax (:481-639, sliding chunks :758-867) over bf16 qkv
 *                              [rows, ld] (rows = [q | k | v], q not yet scaled; ld % 8 == 0; `rows` = the buffer's row count):
 *                              S = Q K^T and O += P V as kind::f16 tcgen05.mma with fp32 accumulation, fp32 softmax, P rounded
 *                              to bf16.  Same masks and padded-query zeros as mts_band_attn_fwd; S <= 4094.  Outputs: out fp32
 *                              [rows, nheads*hd] and / or out_lo [rows, Kp] (the packed operand of mts_gemm_bf16p, Kp ==
 *                              nheads*hd); lse [B, nheads, S] or NULL.  Head dims: those of mts_band_attn_bf16_supported (else
 *                              MTS_E_UNSUPPORTED).
 *   mts_band_attn_bf16_supported : nonzero for the head dims mts_band_attn_fwd_bf16 serves: 16, 32, 64, 112, 128 and 144 .. 256
 *                              in steps of 16. */
int mts_gemm_bf16p_out16(const float *A_lo, const float *B_lo, const float *bias, void *C, int M, int N, int Kp, int64_t ldc,
                         void *stream);
int mts_gemm_bf16p_gelu_pair(const float *A_lo, const float *B_lo, const float *bias, float *C, float *C_lo, int M, int N, int Kp,
                             void *stream);
int mts_embed_ln_fwd_bf16in(const void *x, int64_t x_bstride, const float *pos, const float *typ, const float *gamma,
                            const float *beta, int B, int S, int d, float eps, float *y, float *y_lo, int Kp,
                            const int32_t *lengths, const int32_t *offsets, void *stream);
int mts_band_attn_fwd_bf16(const void *qkv, int64_t ld, int64_t rows, const int32_t *lengths, const int32_t *offsets, int B,
                           int S, int nheads, int hd, int w, float *out, float *out_lo, int Kp, float *lse, void *stream);
int mts_band_attn_bf16_supported(int hd);

/* Profiling hook of the tensor-core recurrence: installs (or, with NULL, removes) a device buffer of 4 x 12 int64
 * into which CTA 0 writes clock64() stamps of the phases of steps 8..11 (see csrc/lstm_rec_tc.cu). */
int mts_debug_rec_profile(long long *buf);

/* The tensor-core recurrence with fp16-split operands (csrc/lstm_rec_h3.cu; nn.LSTM at NeuralArchitectures.py:113-115).
 * W_hh rows (scaled by an exact per-row power of two) and h are each written as two fp16 pieces; W h = W1 h1 + W2 h1 +
 * W1 h2 runs as 48 kind::f16 MMAs per step (relative error ~2^-22), both W pieces resident in tensor memory, and the
 * sender of h_t writes the fp16 pieces straight into the operand buffers of all 8 CTAs of the cluster -- the receivers
 * derive nothing and issue the MMAs of a K-slot as soon as it lands.  Same arguments and results (to fp32 rounding) as
 * mts_lstm_rec_fwd_tc; precision 0 = the fp32-parity path, 1 = one bf16 x bf16 product (the explicit bf16 path). */
int mts_lstm_rec_fwd_h3(const float *gx, const float *w_hh, const int32_t *lengths, const int32_t *order, int n_enc,
                        int B, int T, int H, float *y, float *gates, float *y_corr, int precision, void *stream);
int mts_debug_rec_profile_h3(long long *buf);

/* The fp16-split recurrence with the h tile shared by CTA PAIRS (csrc/lstm_rec_h3p.cu): the two CTAs of a pair issue one
 * M = 256 tcgen05.mma.cta_group::2 stream whose B operand (the 16 episodes' h rows) is split between them, so every CTA
 * receives only half of the rows and every sender addresses 4 CTAs instead of 8 -- half the distributed-shared-memory bytes
 * per step.  Same arguments and results as mts_lstm_rec_fwd_h3. */
int mts_lstm_rec_fwd_h3p(const float *gx, const float *w_hh, const int32_t *lengths, const int32_t *order, int n_enc,
                         int B, int T, int H, float *y, float *gates, float *y_corr, int precision, void *stream);
int mts_debug_rec_profile_h3p(long long *buf);

/* Backward through time of the same layer.
 *   dy      [B, T, n_enc*2H]    gradient w.r.t. y (ignored at t >= len_b)
 *   gates   as saved by the forward call
 *   w_hh_t  [n_enc, 2, H, 4H]   transposed copy of w_hh (row pairs adjacent: feeds the packed-fp32 FMA pipe)
 *   dgx     [n_enc, B*T, 2*4H]  gradient w.r.t. gx (zero at padded steps).  The weight gradients are GEMMs
 *                               over dgx issued by the caller: dW_ih = dgx^T X, dW_hh = dgx^T H_prev
 *                               (mts_gemm_f32 layout 3 with a row shift), db = mts_colsum(dgx).
 */
int mts_lstm_rec_bwd(const float *dy, const float *gates, const float *w_hh, const float *w_hh_t,
                     const int32_t *lengths, const int32_t *order, int n_enc, int B, int T, int H, float *dgx,
                     void *stream);

/* The same backward recurrence on the tensor cores (H == 256 only): the transposed weight slice of every CTA
 * resident in tensor memory, tcgen05.mma per step, partial products reduce-scattered through distributed shared
 * memory.  Same results (to fp32 rounding) as mts_lstm_rec_bwd; needs no transposed copy of w_hh. */
int mts_lstm_rec_bwd_tc(const float *dy, const float *gates, const float *w_hh, const int32_t *lengths,
                        const int32_t *order, int n_enc, int B, int T, int H, float *dgx, void *stream);
/* The same on fp16-split operands (csrc/lstm_bwd_h3.cu): W_hh^T dp = W1 D1 + W2 D1 + W1 D2 as 48 kind::f16 MMAs per step
 * instead of 64 (TF32 + bf16), per-row power-of-two scale of the weight slice and a per-step, per-episode power-of-two scale
 * of dp (column maximum by one warp-wide integer max), both undone in the reduce-scatter epilogue.  The default behind
 * mts_lstm_rec_bwd_tc (MTS_BWD_IMPL=tf32 keeps the TF32 + bf16 kernel); same arguments and results (error ~2^-22 of the
 * column scale). */
int mts_lstm_rec_bwd_h3(const float *dy, const float *gates, const float *w_hh, const int32_t *lengths,
                        const int32_t *order, int n_enc, int B, int T, int H, float *dgx, void *stream);
int mts_lstm_rec_bwd_tf32(const float *dy, const float *gates, const float *w_hh, const int32_t *lengths,
                          const int32_t *order, int n_enc, int B, int T, int H, float *dgx, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Head + decode  (models/CRF.py:340,361-369: Linear then sigmoid/softmax threshold)
 *   feats [B,T,F] (row stride F), w [n_out,F], bias [n_out] -> scores [B,T,n_out];
 *   tags [B,T] uint8 = (n_out==1 ? sigmoid(s) : softmax(s)[1]) > th  for t < len_b, 0xFF beyond.
 *   tags may be NULL (training).  n_out in {1,2}.
 * ---------------------------------------------------------------------------------------------- */
int mts_head_fwd(const float *feats, const float *w, const float *bias, const int32_t *lengths, int B, int T, int F,
                 int n_out, float th, float *scores, uint8_t *tags, void *stream);
/* d_scores [B,T,n_out] -> d_feats [B,T,F], d_w [n_out,F], d_bias [n_out] (all overwritten);
 * ws: >= mts_head_bwd_ws_bytes() bytes of scratch. */
int64_t mts_head_bwd_ws_bytes(int B, int T, int F, int n_out);
int mts_head_bwd(const float *d_scores, const float *feats, const float *w, int B, int T, int F, int n_out,
                 float *d_feats, float *d_w, float *d_bias, void *ws, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Segmentation losses over the valid (un-padded) sentences of a batch (models/CRF.py:342-356).
 *   kind 0: sigmoid focal loss on logits (models/focal_loss.py:38-57), alpha/gamma as given
 *   kind 1: Sigmoid + nn.BCELoss (log clamped at -100)
 *   kind 2: CrossEntropyLoss(ignore_index=-1) on [B*T,2] logits over ALL B*T positions
 *   scores [B,T,n_out]; target [B,*] float with row stride ldt (the collater's tgt_tokens);
 *   inv_count: 1/N with N = sum(lengths) (kinds 0,1) -- passed in so data-parallel ranks can use the
 *   GLOBAL N; kind 2 counts its own non-ignored targets when inv_count <= 0.
 *   loss_out: 2 floats {loss, number of counted positions}.  partial: >= 2*1024 floats of scratch.
 * ---------------------------------------------------------------------------------------------- */
int mts_seg_loss_fwd(const float *scores, const float *target, int64_t ldt, const int32_t *lengths, int B, int T,
                     int kind, float alpha, float gamma, float inv_count, float *loss_out, float *partial,
                     void *stream);
/* d_scores = grad_out * d loss / d scores, zero at padded / ignored positions.  count_dev: device pointer to
 * the count written by the forward call (loss_out + 1), used when inv_count <= 0; may be NULL otherwise. */
int mts_seg_loss_bwd(const float *scores, const float *target, int64_t ldt, const int32_t *lengths, int B, int T,
                     int kind, float alpha, float gamma, float inv_count, const float *count_dev,
                     const float *grad_out, float *d_scores, void *stream);

/* On-device evaluation counts (models/lightning_model.py:16-55, 607-637 walk every episode on the host through
 * segeval).  tags [B, ld_tags] uint8 predictions (mts_head_fwd / Viterbi paths cast to uint8), target [B, ldt] float
 * (the collater's tgt_tokens), lengths int32.  Both sides get their last unit forced to a boundary (as compute_Pk
 * does); `zero_last` first clears it (the end_boundary option).  out [B, 8] int32 =
 *   {Pk mismatches, WindowDiff mismatches, n - k (number of windows), k, tp, fp, fn, reference segments},
 * k = segeval's default window round-half-even(n / (2 segments)), min 2.  The host forms Pk = out0/out2 etc. */
int mts_seg_metrics(const uint8_t *tags, int64_t ld_tags, const float *target, int64_t ldt, const int32_t *lengths,
                    int B, int T, int zero_last, int32_t *out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Linear-chain CRF (models/CRF.py:98-240) on emissions [B,L,C], C = tags + 2 (START = C-2, STOP = C-1),
 * trans[i*C + j] = score of j -> i, lengths int32.  3 <= C <= 8.
 * ---------------------------------------------------------------------------------------------- */
/* Viterbi (CRF.py:172-216): sequential fp32 max-plus recurrence, first maximum wins; on-device back-trace.
 *   best_score [B]; paths [B,L] int32, -1 beyond len_b; bp_ws: B*L uint32 of scratch (packed back-pointers). */
int mts_crf_viterbi(const float *emis, const int32_t *lengths, const float *trans, int B, int L, int C,
                    float *best_score, int32_t *paths, uint32_t *bp_ws, void *stream);
/* NLL pieces (CRF.py:130-170, 218-240): log partition, gold-path score; alphas [B,L,C] saved for backward.
 *   tags [B,*] float (row stride ldt, values in [0, C-2)). */
int mts_crf_nll_fwd(const float *emis, const float *tags, int64_t ldt, const int32_t *lengths, const float *trans,
                    int B, int L, int C, float *log_z, float *gold, float *alphas, void *stream);
/* scale_dev [B]: d loss / d log_z[b] on the device (= -d loss / d gold[b]; grad_out / B for the mean).
 * d_emis [B,L,C] (overwritten, zero at padded steps); d_trans [C,C] (overwritten). */
int mts_crf_nll_bwd(const float *emis, const float *tags, int64_t ldt, const int32_t *lengths, const float *trans,
                    const float *alphas, int B, int L, int C, const float *scale_dev, float *d_emis,
                    float *d_trans, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Pyramidal windowed-attention encoder (HF LongformerModel as driven by
 * models/RestrictedTransformerLayer.py:65-133 and models/CRF.py:521-536; d_model = input width, all-local
 * attention, LayerNorm eps 1e-12, GELU(erf)).  The dense layers are mts_gemm_tf32x3; these are the fused
 * kernels around them.  Every kernel takes `lengths` -- the reference's host-built mask tensors
 * (create_masks_huggingface, RestrictedTransformerLayer.py:101-116) are never materialised.
 *
 * Row layouts.  offsets == NULL: the reference's padded layout, token (b, t) is row b*S + t of every [B*S, .]
 * tensor.  offsets != NULL (int32 [B], offsets[b] = sum of the lengths before b): the RAGGED layout -- only the
 * N = sum(len_b) valid sentences have rows, token (b, t < len_b) is row offsets[b] + t and every token tensor is
 * [N, .].  Padded sentences never influence valid ones (their keys are masked, HF :578-585), so all results at valid
 * positions are identical; the dense layers, LayerNorms and GELU simply run on N instead of B*S rows.  lse / delta
 * keep their [B, nheads, S] shape in both layouts.
 * ---------------------------------------------------------------------------------------------- */
/* LongformerEmbeddings (HF modeling_longformer.py:401-442): y[b,t,:] = LN(x[b,t,:] + pos[t+2,:] + typ[:]).
 *   x [B,S,d] with batch stride x_bstride (elements); pos = the full position table [>= S+2, d]; d % 4 == 0.
 *   y [B*S,d]; optional y_hi/y_lo [B*S,Kp] = the operand pair of y for the next GEMM; y_hi may be NULL when Kp == d
 *   (y itself is then the `hi` operand: no duplicate write);
 *   optional sum_out [B*S,d] (pre-LN values) and stats [B*S,2] = (mean, rstd), saved for the backward pass.
 *   lengths/offsets (both or neither): write the outputs in the ragged layout (x stays [B,S,d]). */
int mts_embed_ln_fwd(const float *x, int64_t x_bstride, const float *pos, const float *typ, const float *gamma,
                     const float *beta, int B, int S, int d, float eps, float *y, float *y_hi, float *y_lo, int Kp,
                     float *sum_out, float *stats, const int32_t *lengths, const int32_t *offsets, void *stream);
/* LongformerSelfOutput / LongformerOutput (:1060-1071, :1119-1130): y = LN(a + res); a is the dense output
 *   (bias already added by the GEMM epilogue).  sum_out may alias a.  res may be NULL: a then already holds the
 *   sum (the dense layer accumulated onto the residual in its epilogue: mts_gemm_tf32x3 with accumulate = 1), which
 *   spares this kernel one of its two input reads. */
int mts_add_ln_fwd(const float *a, const float *res, const float *gamma, const float *beta, int M, int d, float eps,
                   float *y, float *y_hi, float *y_lo, int Kp, float *sum_out, float *stats, void *stream);
/* The same two LayerNorms writing, next to y, the FP16-SPLIT operand of mts_gemm_f16x3 instead of the (hi, lo) pair:
 *   pieces [rows][2][K64] fp16 (K64 % 64 == 0, zero beyond d): fp16(y s) and fp16(y s - fp16(y s)), s = the exact power of two
 *   that puts the row's largest |y| into [2^13, 2^14); row_scale [rows] = 1 / s.  d <= 1024.  Inference only (no saved tensors). */
int mts_embed_ln_fwd_f16(const float *x, int64_t x_bstride, const float *pos, const float *typ, const float *gamma,
                         const float *beta, int B, int S, int d, float eps, float *y, void *pieces, int K64, float *row_scale,
                         const int32_t *lengths, const int32_t *offsets, void *stream);
int mts_add_ln_fwd_f16(const float *a, const float *res, const float *gamma, const float *beta, int M, int d, float eps, float *y,
                       void *pieces, int K64, float *row_scale, void *stream);
/* The embeddings LayerNorms over an early-fusion PAIR read in place: x[b, t, :] = [src1[b, t, :D1] | src2[b, t, :D2]], each
 * source [B, S, D_i] with dense rows (row pitch D_i) and its own batch stride bstride_i (elements), d = D1 + D2.  Every output,
 * and every other argument, as in mts_embed_ln_fwd / mts_embed_ln_fwd_f16 / mts_embed_ln_fwd_bf16in for the concatenated
 * tensor, bit for bit.  D1 % 4 == 0, D2 % 4 == 0; sources on 16 bytes (fp32) or 8 bytes (bf16), bstride_i % 4 == 0; otherwise
 * MTS_E_UNSUPPORTED (concatenate and call the single-source entry). */
int mts_embed_ln_fwd_pair(const float *src1, int64_t bstride1, int D1, const float *src2, int64_t bstride2, int D2,
                          const float *pos, const float *typ, const float *gamma, const float *beta, int B, int S, float eps,
                          float *y, float *y_hi, float *y_lo, int Kp, float *sum_out, float *stats, const int32_t *lengths,
                          const int32_t *offsets, void *stream);
int mts_embed_ln_fwd_f16_pair(const float *src1, int64_t bstride1, int D1, const float *src2, int64_t bstride2, int D2,
                              const float *pos, const float *typ, const float *gamma, const float *beta, int B, int S, float eps,
                              float *y, void *pieces, int K64, float *row_scale, const int32_t *lengths, const int32_t *offsets,
                              void *stream);
int mts_embed_ln_fwd_bf16in_pair(const void *src1, int64_t bstride1, int D1, const void *src2, int64_t bstride2, int D2,
                                 const float *pos, const float *typ, const float *gamma, const float *beta, int B, int S,
                                 float eps, float *y, float *y_lo, int Kp, const int32_t *lengths, const int32_t *offsets,
                                 void *stream);
/* LongformerIntermediate (:1103-1116) activation fused with the operand split: hi/lo [rows,Kp] of GELU(src);
 * act [rows,cols] or NULL: GELU(src) in fp32, kept for the weight gradient of the next dense layer. */
int mts_gelu_split(const float *src, int64_t ld, int rows, int cols, int Kp, float *act, float *hi, float *lo,
                   void *stream);
/* LongformerSelfAttention (:481-639; sliding chunks :758-867) for all-local attention:
 *   qkv [B*S, ld] rows = [q | k | v] (each nheads*hd wide, head-major), q NOT yet scaled (the kernel divides by
 *   sqrt(hd) as HF does at :513); token i attends to j with |i-j| <= w and j < len_b; softmax in fp32;
 *   rows i >= len_b give exact zeros (:578).  hd % 4 == 0, hd <= 256.
 *   out [B*S, nheads*hd] and/or its TF32 halves out_hi/out_lo [B*S,Kp] (Kp == nheads*hd);
 *   lse [B,nheads,S] or NULL: log-sum-exp of every query row, saved for the backward pass. */
int mts_band_attn_fwd(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B, int S,
                      int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp, float *lse,
                      void *stream);
/* The same on the tensor cores: warp-level mma.sync m16n8k8 TF32 with 3xTF32 compensation for Q K^T and P V, S kept in
 * registers (hd in {8,16,32,64,112,128}).  Same contract and results; on B200 it runs at the speed of the CUDA-core
 * kernel (measured).  Kept as a second implementation; MTS_ATTN_IMPL=mma switches the default entry over to it. */
int mts_band_attn_fwd_mma(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B, int S,
                          int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp, float *lse,
                          void *stream);
/* The CUDA-core (packed FFMA2) kernel: any head dim that is a multiple of 4 and <= 256.  mts_band_attn_fwd falls back
 * to it for head dims the tcgen05 kernel is not instantiated for (among them every head dim above 128). */
int mts_band_attn_fwd_simt(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B, int S,
                           int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp, float *lse,
                           void *stream);
/* The tcgen05 kernel (csrc/attn_tc.cu), the default behind mts_band_attn_fwd: Q K^T and P V as tcgen05.mma (TF32 +
 * packed bf16 correction, both operands' corrections derived on chip), S / P / O in tensor memory, fp32 softmax from
 * tcgen05.ld.  Replaces HF's sliding-chunk einsums (modeling_longformer.py:758-867; call site
 * models/RestrictedTransformerLayer.py:131).  Head dims 16, 32, 64, 112, 128 (mts_band_attn_tc_supported). */
int mts_band_attn_tc_supported(int hd);
/* development hook: a device buffer of 6 x 5 x 40 int64 receives clock64() stamps of CTA 0's first work items (NULL: off) */
int mts_debug_attn_profile(long long *buf);
int mts_band_attn_fwd_tc(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B, int S,
                         int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp, float *lse,
                         void *stream);

/* Backward of the encoder pieces (the reference: autograd through HF LongformerModel).
 * mts_ln_bwd: dy, pre (pre-LN values), stats (mean, rstd) as saved by the forward calls -> dx [M,d] (+ its TF32
 *   operand pair dx_hi/dx_lo [M,Kp]; dx_hi may be NULL when Kp == d), dgamma [d], dbeta [d] (overwritten);
 *   ws >= mts_ln_bwd_ws_bytes. */
int64_t mts_ln_bwd_ws_bytes(int M, int d);
int mts_ln_bwd(const float *dy, const float *pre, const float *stats, const float *gamma, int M, int d, float *dx,
               float *dx_hi, float *dx_lo, int Kp, float *dgamma, float *dbeta, void *ws, void *stream);
/* dzp = dz * GELU'(zp) [rows,cols] and its TF32 halves hi/lo [rows,Kp]. */
int mts_gelu_bwd(const float *dz, const float *zp, int rows, int cols, int Kp, float *dzp, float *hi, float *lo,
                 void *stream);
/* dpos[t,:] = sum_b dpre[b,t,:]  (gradient rows 2..S+1 of the position table; the token-type gradient is the
 * column sum of dpos, mts_colsum). */
int mts_embed_bwd(const float *dpre, int B, int S, int d, float *dpos, const int32_t *lengths, const int32_t *offsets,
                  void *stream);
/* Banded attention backward: qkv, lse as in the forward call, o = forward output [B*S, nheads*hd], d_o its
 * gradient -> dqkv [B*S, ld] = [dq | dk | dv] (dq already includes the 1/sqrt(hd) factor), zero at padded rows.
 * delta_ws: B*nheads*S floats of scratch.  hd % 4 == 0, hd <= 256. */
int mts_band_attn_bwd(const float *qkv, int64_t ld, const float *o, const float *d_o, const float *lse,
                      const int32_t *lengths, const int32_t *offsets, int B, int S, int nheads, int hd, int w, float *dqkv,
                      float *delta_ws, void *stream);
/* Training with dropout on the attention probabilities -- HF `attention_probs_dropout_prob`, set by the reference from
 * `dropout_out` (models/CRF.py:531-536 -> models/RestrictedTransformerLayer.py:85-92; `nn.functional.dropout(attn_probs)`
 * in modeling_longformer.py LongformerSelfAttention.forward).  Same contracts as mts_band_attn_fwd_simt / mts_band_attn_bwd
 * with P V weighted by p * keep / (1 - p_drop); `lse` stays the log-sum-exp of the undropped scores.  keep(b, head, i, j)
 * is a pure function of `seed` and the indices (csrc/common.cuh attn_keep_scale; oracle/ref_numpy.py attn_dropout_keep is
 * its numpy restatement), so the backward call regenerates the forward mask from the same seed: no mask tensor.
 * p_drop in [0, 1); p_drop == 0 is the plain kernel. */
int mts_band_attn_fwd_dropout(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B, int S,
                              int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp, float *lse,
                              float p_drop, uint64_t seed, void *stream);
int mts_band_attn_bwd_dropout(const float *qkv, int64_t ld, const float *o, const float *d_o, const float *lse,
                              const int32_t *lengths, const int32_t *offsets, int B, int S, int nheads, int hd, int w,
                              float *dqkv, float *delta_ws, float p_drop, uint64_t seed, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MTS_B200_H_ */
