/* pm_emage.h - C ABI of libpm_emage.so: the B200 (sm_100a) kernels of the EMAGE audio->motion
 * inference hot path.
 *
 * The reference (PantoMatrix) has no FFI for this path: every op below is a stock torch.nn /
 * torch.nn.functional call made from Python (SURVEY.md section 8b).  Each entry point therefore
 * cites the reference *call site* it replaces; the Python modules in pantomatrix_b200/emage_audio
 * (same names and signatures as /root/reference/models/emage_audio/__init__.py:1-12) are the only
 * callers.  M.py = models/emage_audio/modeling_emage_audio.py, P.py = .../processing_emage_audio.py.
 *
 * Conventions
 *   - plain pointers + explicit sizes; all pointers are DEVICE pointers unless noted
 *   - activations are channels-last fp32: tensor (batch, rows, channels), row stride `ld*` in elements,
 *     batch stride `*_bs` in elements (lets callers pass column slices / overlapping windows)
 *   - `stream` is a cudaStream_t passed as void*; nothing allocates, nothing synchronises
 *   - return 0 = ok, <0 = PM_E* argument error, >0 = cudaError_t from the launch
 *   - optional split-bf16 output (`planes`, p_ps, p_ld, p_nsplit): the producer also (or only, when its fp32
 *     `out` is NULL) writes its result as p_nsplit bf16 planes (x ~ p0+p1+p2, plane stride p_ps, row stride
 *     p_ld elements): the A operand format of pm_tapgemm_tc, so no separate conversion pass is needed
 *   - plane element format: bit 8 (PM_FMT_F16) of any `nsplit` / `p_nsplit` / `out_nsplit` argument selects IEEE fp16
 *     planes instead of bf16 (same 2-byte storage).  Two fp16 planes carry 22 mantissa bits, so nsplit = 2
 *     (3 tensor-core products) gives the accuracy of 3 bf16 planes (6 products) - provided magnitudes stay below
 *     65504; an overflow becomes inf - inf = NaN in the consuming GEMM, which the host checks for.
 */
#ifndef PM_EMAGE_H
#define PM_EMAGE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define PM_ABI_VERSION 5
#define PM_FMT_F16 0x100
int pm_abi_version(void);
/* cudaMemsetAsync on `stream` (a memset node under graph capture, not a kernel): zeroed slack rows, flags */
int pm_memset_async(void* ptr, int value, long long bytes, void* stream);
/* compute capability major*10+minor of the current device, or <0 */
int pm_device_cc(void);

/* ---- tap-GEMM: Conv1d (any kernel size/stride/zero padding) and Linear as one op ------------------
 * out[b,l,n] = act( bias[n] + sum_{t<taps} sum_{c<cin} A[b, l*stride + t - pad, c] * W[t,n,c]
 *                   + residual[b,l,n] ),  rows of A outside [0,rows_in) read as zero.
 * W is (taps, cout, cin) fp32 (BatchNorm already folded in by the host packer).
 * Replaces: nn.Conv1d+BatchNorm1d+LeakyReLU(+shortcut add) in BasicBlock P.py:283-294, the k=3 convs of
 * ResBlock/VQEncoderV6/VQDecoderV5 P.py:178-261, nn.Linear everywhere (MLP P.py:322-326, projections
 * M.py:288,293,297,304,323-325, MultiheadAttention in/out projections and FFN linear1/linear2 inside
 * nn.Transformer{En,De}coderLayer M.py:238-250).  fp32 SIMT reference engine (exact-order fp32 FMA). */
int pm_tapgemm_f32(const float* A, long long a_bs, int lda, int batch, int rows_in, int cin,
                   const float* W, const float* bias, int taps, int stride, int pad,
                   int rows_out, int cout,
                   const float* residual, long long r_bs, int ldr,
                   int act, float slope,
                   float* out, long long o_bs, int ldo, void* stream);

/* ---- tap-GEMM on the tcgen05 tensor cores (split-bf16 operands, fp32 TMEM accumulate) -------------
 * Same contract as pm_tapgemm_f32 with stride == 1 (strided convs are passed as stride-1 problems over the
 * (rows/s, s*cin) view of the input with zero-padded taps).  A and W are `nsplit` bf16 planes (x = p0+p1+p2),
 * plane strides a_ps / w_ps elements: nsplit 1 = plain bf16, 2 = bf16x3 (p0*p0 + p0*p1 + p1*p0), 3 = bf16x6
 * (all products down to 2^-24).  W planes are (taps, w_rows, ldw) with w_rows >= cout a multiple of the N
 * tile (64 if cout <= 64 else 128), zero rows beyond cout.  lda, ldw, a_bs, a_ps, w_ps must be multiples
 * of 8 elements (TMA 16-byte rule).  The activation is applied to columns < act_cols only (<=0: all).
 * The epilogue writes the fp32 result and/or its bf16 split planes (out_f32 / out_bf16 nullable).
 * Operands are staged by TMA (cp.async.bulk.tensor, zero fill for padding rows, tap shift folded into the
 * row coordinate); descriptors are built on the host inside this call from the raw pointers.
 * `prefetch` (nullable, 16-byte aligned): prefetch_bytes of global memory - the NEXT GEMM's packed weights - are
 * pulled into L2 by this launch (cp.async.bulk.prefetch.L2), so weight streaming overlaps the previous GEMM.
 * fp16 operands (nsplit | PM_FMT_F16): the host packs W scaled by a power of two into the top of the fp16 range;
 * `acc_scale` (its reciprocal, exact) multiplies the accumulator before bias.  Must be 1 for bf16 operands. */
int pm_tapgemm_tc(const uint16_t* A, long long a_ps, long long a_bs, int lda, int batch, int rows_in, int cin,
                  const uint16_t* W, long long w_ps, int w_rows, int ldw, int taps, int pad, int nsplit,
                  const float* bias, int rows_out, int cout,
                  const float* residual, long long r_bs, int ldr,
                  int act, int act_cols, float slope, float acc_scale,
                  float* out_f32, long long o_bs, int ldo,
                  uint16_t* out_bf16, long long ob_ps, long long ob_bs, int ldob, int out_nsplit,
                  const void* prefetch, long long prefetch_bytes, void* stream);

/* fp32 (batch, rows, ch) -> nsplit bf16 planes (round-to-nearest hi, then residual planes). */
int pm_split_bf16(const float* x, long long x_bs, int ldx, int batch, int rows, int ch,
                  uint16_t* out, long long o_ps, long long o_bs, int ldo, int nsplit, void* stream);

/* ---- WavEncoder stem: first BasicBlock's conv1 and downsample conv on the raw waveform (Cin = 1) --
 * sequence (b, w) starts at audio + b*a_bs + w*a_ws and is n_samples long; k=15, stride 5, pad 1600.
 * Outputs are window-major: row block (w*batch + b) of (windows*batch, rows_out, cout).
 * y1 = LeakyReLU_0.01(conv1*bn1), sc = downsample conv*bn (both BN-folded): P.py:285-291,301.
 * y1 goes out as fp32 (`y1`, nullable) and / or as the next GEMM's operand planes (`planes`, nullable; dense rows of
 * p_ld elements, plane stride p_ps, p_nsplit | PM_FMT_F16 as for pm_add_layernorm_f32); at least one of the two.
 * cout 32 or 64, ksize 15; anything else returns PM_EUNSUPPORTED. */
int pm_wav_stem_f32(const float* audio, long long a_bs, long long a_ws, int batch, int windows, int n_samples,
                    const float* w1, const float* b1, const float* wd, const float* bd, int cout,
                    int ksize, int stride, int pad, int rows_out, float slope,
                    float* y1, float* sc,
                    uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream);

/* ---- LayerNorm(x + r) * gamma + beta over the last dim (r nullable): post-norm residual of
 * nn.TransformerEncoderLayer / DecoderLayer (M.py:238-250), eps 1e-5.  ch must be a multiple of 128 <= 1024 */
int pm_add_layernorm_f32(const float* x, const float* r, const float* gamma, const float* beta,
                         float* out, long long rows, int ch, float eps,
                         uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream);

/* ---- multi-head attention core, no masks: softmax(Q K^T / sqrt(hd)) V for Tq,Tk <= 64, hd = 192 ----
 * Q/K/V rows are (b*T + t) with row strides ldq/ldk/ldv; head h occupies columns [h*hd,(h+1)*hd).
 * Replaces scaled_dot_product_attention inside nn.MultiheadAttention (M.py:238-250 layers). */
int pm_attention_f32(const float* Q, int ldq, const float* K, int ldk, const float* V, int ldv,
                     float* O, int ldo, int batch, int heads, int tq, int tk, int head_dim,
                     uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream);

/* Same op on the tcgen05 tensor cores for the fp16x3 engine: Q, K, V are two-plane fp16 activations (x = (p0+p1)/64,
 * plane stride *_ps, clip stride *_bs, row stride ld* elements, *_cols valid columns; head h of Q starts at column
 * q_col0 + h*hd, likewise K and V - so the packed q|k|v projection output is consumed in place through TMA).
 * S = Q K^T and O = P V run as 3-product fp16 UMMAs (M=64) with S and O in TMEM, softmax in fp32 registers.
 * Output: fp32 O (nullable) and / or two fp16 planes (p_nsplit = 2 | PM_FMT_F16). */
int pm_attention_tc(const uint16_t* Q, long long q_ps, long long q_bs, int ldq, int q_cols, int q_col0,
                    const uint16_t* K, long long k_ps, long long k_bs, int ldk, int k_cols, int k_col0,
                    const uint16_t* V, long long v_ps, long long v_bs, int ldv, int v_cols, int v_col0,
                    float* O, int ldo, int batch, int heads, int tq, int tk, int head_dim,
                    uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream);

/* ---- broadcast adds: out[b,t,:] = ((x[b,t,:] + first) + second), each of first/second chosen by code:
 * 0 = nothing, 1 = pe[t,:] (PeriodicPositionalEncoding P.py:341-343), 2 = spk[b,:] (speaker embedding
 * row repeated over t, M.py:285-286).  x nullable (treated as 0).  Preserves the reference's add order
 * (M.py:291,298-299,307-308,320-322). */
int pm_add_rows_f32(const float* x, const float* pe, const float* spk, int first, int second,
                    float* out, int batch, int rows, int ch,
                    uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream);
/* out = a + b over n elements viewed as rows of `ch` (M.py:312,320-325) */
int pm_add2_f32(const float* a, const float* b, float* out, long long n, int ch,
                uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream);

/* ---- window assembly (M.py:384-391 and 267-268 fused): builds one window's motion-encoder input.
 * motion/mask: (batch, total_len, ch) full-sequence tensors, either may be NULL = inference()'s defaults (identity
 * rot6d + zero trans/contact; all masked, M.py:369-377); seed: (batch, pre, ch) decoded last frames, clip stride seed_bs.
 * For frame f<pre: v = mask==0 ? motion : seed (seed NULL = the first window, whose seed is motion[:, :pre] itself,
 * M.py:379), window mask forced 0; else v = motion, m = mask.
 * out = (m == 1) ? mask_embedding[c] : v. */
int pm_window_input_f32(const float* motion, const float* mask, const float* seed, const float* mask_embedding,
                        float* out, int batch, int total_len, int start, int win_len, int pre, int ch, long long seed_bs,
                        uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream);

/* ---- VQ ------------------------------------------------------------------------------------------ */
/* index = argmin_k ( |z|^2 + |e_k|^2 - 2 z.e_k ) evaluated in fp32, first minimum wins (a row of NaNs yields 0, like
 * torch.argmin): EmageVQVAEConv.decode_from_latent M.py:60-65, Quantizer.map2index P.py:158-164.
 * e2 = precomputed |e_k|^2 (n_codes).  Writes int64 indices.  e_dim must be 256.
 *   pm_l2_argmin_tc      n_codes == 256: persistent tcgen05 kernel - fp16 UMMA screen of all 256 scores per row with a
 *                        rigorous error bound, exact fp32 re-scoring of every row whose best two screened distances
 *                        are within that bound; each z row is read from HBM once (1 KB + 8 B written per row).
 *                        max_ctas > 0 caps the persistent grid (<= 0: one CTA per SM).
 *   pm_l2_argmin_simt_f32  n_codes a multiple of 64: register-tiled fp32 SIMT kernel (sequential-k fp32 FMA).
 *   pm_l2_argmin_f32     dispatcher the product calls: tc for 256-code codebooks, simt otherwise. */
int pm_l2_argmin_f32(const float* z, long long rows, int rows_per_batch, long long z_bs,
                     const float* codebook, const float* e2, int n_codes, int e_dim, long long* index, void* stream);
int pm_l2_argmin_tc(const float* z, long long rows, int rows_per_batch, long long z_bs,
                    const float* codebook, const float* e2, int n_codes, int e_dim, long long* index, int max_ctas,
                    void* stream);
int pm_l2_argmin_simt_f32(const float* z, long long rows, int rows_per_batch, long long z_bs,
                          const float* codebook, const float* e2, int n_codes, int e_dim, long long* index, void* stream);
/* index = first argmax over the last dim: torch.max(F.log_softmax(x,2),2)[1], M.py:398-401 (monotone).
 * Row r of the (batch, rows_per_batch, ch) view lives at x + (r / rows_per_batch)*x_bs + (r % rows_per_batch)*ldx
 * (rows_per_batch <= 0: one dense matrix; the same convention addresses z in pm_l2_argmin_* with ld = 256), so the
 * tail frames of a window are read in place.  nonfinite (nullable): set to 1 when any element read is NaN / inf. */
int pm_row_argmax_f32(const float* x, long long rows, int ch, int ldx, int rows_per_batch, long long x_bs,
                      long long* index, int* nonfinite, void* stream);
/* out[r,:] = codebook[index[r],:]: Quantizer.get_codebook_entry P.py:166-170, nn.Embedding M.py:285-286.
 * n_table = rows of `codebook`; indices outside [0, n_table) are clamped (never an out-of-bounds read). */
int pm_gather_rows_f32(const float* codebook, long long n_table, const long long* index, long long rows, int ch,
                       float* out, uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream);
/* |e_k|^2 per codebook row (done once at pack time) */
int pm_row_sqnorm_f32(const float* x, int rows, int ch, float* out, void* stream);

/* ---- pose composition: EmageVQModel.decode M.py:135-188 + rotation conversions P.py:6-104 ---------
 * face (bt,106) | upper (bt,78) | hands (bt,180) | lower (bt,61) decoder outputs (any may be NULL = the
 * reference's zero branch) -> expression (bt,100), axis_angle (bt,165), motion4inf (bt,337). */
int pm_pose_compose_f32(const float* face, const float* upper, const float* hands, const float* lower,
                        float* expression, float* axis_angle, float* motion4inf, long long bt, void* stream);

/* ---- global translation: velocity2position P.py:107-115 as used by get_global_motion M.py:195-205 --
 * rec (batch, t, ld) global-AE output; vel = rec[..., 54:57]; x/z integrated sequentially with dt,
 * y copied; ref_trans (batch,3) start position. */
int pm_global_trans_f32(const float* rec, int ld, int vel_off, const float* ref_trans, int ref_bs, float dt,
                        float* trans, int batch, int t, void* stream);

/* ---- ragged batches: clips of different lengths laid out at one capacity ----------------------------------------
 * Each entry point below is the one of the same name without `_rl`, plus per-clip limits, and runs the same kernel
 * (a NULL limit is that entry point).  They keep one invariant, which makes a clip's result in a ragged batch equal
 * its result alone: no kernel that mixes rows (convolution, attention) ever reads a padded row as data.  Limit
 * tables are DEVICE int32 arrays, so a captured graph reads whatever the caller copied into them before a replay.
 *   pm_tapgemm_tc_rl / pm_tapgemm_f32_rl  output row r of clip c is computed as usual if r < row_limit[c]; otherwise
 *       its fp32 and plane outputs are stored as 0 (bias and residual are not read) - the zero padding the next
 *       convolution expects - and a NEGATIVE limit leaves all rows of the clip unwritten.  The clip of output row
 *       (b, l) is b when rows_per_clip == 0, else (b*rows_out + l) / rows_per_clip with row r = the remainder (a
 *       Linear over all clips as one tall matrix).
 *   pm_wav_stem_rl       sequence s (window-major, w*batch + b) holds n_valid[s] <= n_samples samples: later samples
 *       read as 0 (the right-hand zero padding) and rows >= (n_valid + 2*pad - ksize)/stride + 1 are written as 0
 *       (all rows for n_valid == 0).
 *   pm_attention_tc_rl / pm_attention_f32_rl  keys >= k_len[b] get probability 0; query rows >= q_len[b] are written as
 *       0, and so is every row of a clip with k_len[b] == 0.
 *   pm_window_input_rl   rows >= win_len_valid[b] are written as 0.
 *   pm_gather_rows_rl    row r belongs to clip r / rows_per_clip (> 0); rows with r % rows_per_clip >= row_limit[clip]
 *       are written as 0. */
int pm_tapgemm_tc_rl(const uint16_t* A, long long a_ps, long long a_bs, int lda, int batch, int rows_in, int cin,
                     const uint16_t* W, long long w_ps, int w_rows, int ldw, int taps, int pad, int nsplit,
                     const float* bias, int rows_out, int cout,
                     const float* residual, long long r_bs, int ldr,
                     int act, int act_cols, float slope, float acc_scale,
                     float* out_f32, long long o_bs, int ldo,
                     uint16_t* out_bf16, long long ob_ps, long long ob_bs, int ldob, int out_nsplit,
                     const void* prefetch, long long prefetch_bytes, const int* row_limit, int rows_per_clip,
                     void* stream);
int pm_tapgemm_f32_rl(const float* A, long long a_bs, int lda, int batch, int rows_in, int cin,
                      const float* W, const float* bias, int taps, int stride, int pad,
                      int rows_out, int cout,
                      const float* residual, long long r_bs, int ldr,
                      int act, float slope,
                      float* out, long long o_bs, int ldo, const int* row_limit, int rows_per_clip, void* stream);
int pm_wav_stem_rl(const float* audio, long long a_bs, long long a_ws, int batch, int windows, int n_samples,
                   const float* w1, const float* b1, const float* wd, const float* bd, int cout,
                   int ksize, int stride, int pad, int rows_out, float slope,
                   float* y1, float* sc,
                   uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* n_valid, void* stream);
int pm_attention_tc_rl(const uint16_t* Q, long long q_ps, long long q_bs, int ldq, int q_cols, int q_col0,
                       const uint16_t* K, long long k_ps, long long k_bs, int ldk, int k_cols, int k_col0,
                       const uint16_t* V, long long v_ps, long long v_bs, int ldv, int v_cols, int v_col0,
                       float* O, int ldo, int batch, int heads, int tq, int tk, int head_dim,
                       uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* q_len, const int* k_len,
                       void* stream);
int pm_attention_f32_rl(const float* Q, int ldq, const float* K, int ldk, const float* V, int ldv,
                        float* O, int ldo, int batch, int heads, int tq, int tk, int head_dim,
                        uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* q_len, const int* k_len,
                        void* stream);
int pm_window_input_rl(const float* motion, const float* mask, const float* seed, const float* mask_embedding,
                       float* out, int batch, int total_len, int start, int win_len, int pre, int ch, long long seed_bs,
                       uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* win_len_valid, void* stream);
int pm_gather_rows_rl(const float* codebook, long long n_table, const long long* index, long long rows, int ch,
                      float* out, uint16_t* planes, long long p_ps, int p_ld, int p_nsplit,
                      const int* row_limit, int rows_per_clip, void* stream);

/* ---- CaMN / DisCo (BASELINE configs[2],[3]) ------------------------------------------------------- */
/* One bidirectional nn.LSTM layer, zero initial state (camn:205-217,264-271; disco:212-216,255).  xproj (batch, t,
 * ldx >= 8*hidden) holds W_ih x + b_ih + b_hh for both directions (column dir*4H + gate*H + unit, gates i,f,g,o);
 * whh (2, 4H, H) fp32; y (batch, t, ldy >= 2H) receives [forward h | backward h].  `barrier` = 4 uint32 of scratch.
 * hidden must be 512.  Persistent cooperative kernel, W_hh resident in shared memory. */
int pm_lstm_bidir_f32(const float* xproj, long long x_bs, int ldx, const float* whh,
                      float* y, long long y_bs, int ldy, unsigned int* barrier,
                      int batch, int t, int hidden, void* stream);
/* rot6d (rows, n_sel*6) of the selected joints -> axis-angle (rows, 165), zeros at unselected joints: camn:274-277.
 * slot: device int32[55], position of joint j among the selected ones or -1. */
int pm_rot6d_to_aa_f32(const float* rot6d, long long rows, int n_sel, const int* slot, float* out, void* stream);
/* DisCo content mix disco:250-251: out[r,:] = softmax(sel[r,0:2])[0]*c1[r,:] + [1]*c2[r,:] (out row stride ldo) */
int pm_softmax2_mix_f32(const float* sel, const float* c1, const float* c2, float* out, long long rows, int ch, int ldo,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif
