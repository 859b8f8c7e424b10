/* speech_b200 — C ABI of the B200-native (sm_100a) hot path of awni/speech.
 *
 * Boundary rules (SURVEY.md §8b):
 *   - plain C symbols, raw pointers and sizes, no torch / C++ types in any signature;
 *   - every buffer is caller-owned (PyTorch allocates); the library never allocates device
 *     memory, never synchronises the device, and never throws: each entry point returns an
 *     int status (SB_OK == 0) and enqueues its kernels on the cudaStream_t passed as `stream`
 *     (a void* so that this header needs no CUDA include);
 *   - unless stated otherwise every pointer is a DEVICE pointer;
 *   - re-entrant across streams; one process per GPU.
 *
 * Each entry point cites the reference interface it replaces (paths relative to the
 * reference tree, awni/speech @ a5909a3).
 */
#ifndef SPEECH_B200_H_
#define SPEECH_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB_OK 0
#define SB_ERR_INVALID 1      /* bad argument */
#define SB_ERR_CUDA 2         /* a CUDA runtime / driver call failed */
#define SB_ERR_UNSUPPORTED 3  /* shape outside what the kernels implement */
#define SB_ERR_WORKSPACE 4    /* caller-provided workspace too small */

/* library / device introspection -------------------------------------------------------- */
int sb_version(void);                 /* 100 * major + minor */
const char* sb_status_string(int status);
int sb_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* l2_bytes);

/* ---------------------------------------------------------------------------------------
 * CTC loss + gradient.
 * Replaces: functions.ctc.CTCLoss()(acts, labels, act_lens, label_lens)
 *           (libs/warp-ctc pytorch_binding; call site speech/models/ctc_model.py:34-40;
 *            un-vendored dependency cloned by Makefile:4-7).
 *   acts        (B, T, V) float32, batch-first, UN-normalised (softmax is internal)
 *   grads       (B, T, V) float32 out: d(sum_b cost_b)/d acts; may be NULL (costs only)
 *   labels      flat int32 [sum(label_lens)], label_offsets = exclusive prefix sum of label_lens
 *   act_lens    (B) int32 valid frames per utterance (reference passes T for all,
 *               ctc_model.py:43-45); rows >= act_lens[b] get zero gradient
 *   blank       blank class index (reference: V-1, ctc_model.py:18)
 *   costs       (B) float32 out: -log p(labels_b | acts_b); +inf when no alignment exists
 *   workspace   >= sb_ctc_workspace_size(...) bytes
 * ------------------------------------------------------------------------------------- */
int sb_ctc_workspace_size(int B, int T, int V, int max_label_len, size_t* bytes);
int sb_ctc_fwd_bwd(const float* acts, float* grads, const int* labels, const int* label_offsets,
                   const int* label_lens, const int* act_lens, int B, int T, int V, int blank,
                   int max_label_len, float* costs, void* workspace, size_t workspace_bytes,
                   void* stream);

/* ---------------------------------------------------------------------------------------
 * Dense contraction on tcgen05 tensor cores:
 *     C[M,N] (f32)  (+)=  A[M,K] (bf16, row-major) * B[N,K]^T (bf16, row-major)  (+ bias[N])
 * Replaces: the cuBLAS/cuDNN GEMMs reached through nn.GRU / nn.Linear
 *           (speech/models/model.py:35-39, 115-133).
 *   lda/ldb/ldc  leading dimensions in ELEMENTS; A and B rows must be 16-byte aligned
 *   flags        SB_GEMM_ACCUMULATE: C += (atomic adds; required when split_k > 1)
 *                SB_GEMM_ROW_REMAP : row m = t*remap_B + b is stored at row b*remap_T + t
 *                                    (time-major -> batch-first), rows with b >= valid_B dropped
 *                SB_GEMM_A_MN      : A is given as [K][M] (lda = elements per K row; M contiguous)
 *                SB_GEMM_B_MN      : B is given as [K][N] (ldb = elements per K row; N contiguous)
 *                                    -- the contraction runs over the ROWS of the matrix, which is
 *                                    how activations [tokens][features] enter a weight gradient
 *                                    (dW = dY^T X): no transposed copies are needed
 * ------------------------------------------------------------------------------------- */
#define SB_GEMM_ACCUMULATE 1
#define SB_GEMM_ROW_REMAP 2
#define SB_GEMM_A_MN 4
#define SB_GEMM_B_MN 8
int sb_gemm_bf16_tn(const void* A, long long lda, const void* B, long long ldb, float* C,
                    long long ldc, const float* bias, int M, int N, int K, int flags, int split_k,
                    int remap_B, int remap_T, int valid_B, void* stream);

/* ---------------------------------------------------------------------------------------
 * GRU recurrence (T-serial part of nn.GRU; the time-batched input projection is sb_gemm_bf16_tn).
 * Replaces: cuDNN RNN behind self.rnn in speech/models/model.py:35-39,73 (gate order r,z,n;
 *           bidirectional) and Transducer.dec_rnn, speech/models/transducer_model.py:23-26,68.
 * Internal layout is TIME-MAJOR with the batch padded to a multiple of 8: row m = t*Bp + b.
 *   gi     [T*Bp][ndir*3H] f32   X W_ih^T + b_ih (forward-direction gates first)
 *   whh    [ndir][3H][H]   bf16  recurrent weights;   bhh [ndir][3H] f32
 *   y      [T*Bp][ndir*H]  f32   h_t (out)
 *   xn     [T*Bp][ndir*H]  bf16  h_t (out; operand of the next projection and of dW_hh)
 *   gates  [T*Bp][ndir][4][H] f32 saved r,z,n,(W_hn h + b_hn) for backward (out; may be NULL)
 *   workspace  >= sb_gru_fwd_workspace_size bytes, 1024-byte aligned: per-chunk ready counters
 *          and the double-buffered exchange tiles of h_t (zeroed by the call itself)
 * Constraints: H % 16 == 0, Bp % 8 == 0, Bp <= 128, ndir*H/16 <= number of SMs.
 * ------------------------------------------------------------------------------------- */
int sb_gru_fwd_workspace_size(int Bp, int H, int ndir, size_t* bytes);
int sb_gru_fwd(const float* gi, const void* whh_bf16, const float* bhh, float* y, void* xn_bf16,
               float* gates, void* workspace, size_t workspace_bytes, int T, int Bp, int H,
               int ndir, void* stream);

/* "Parity mode" forward recurrence: the same time loop in plain fp32 on CUDA cores (fp32 weights
 * [ndir][3H][H], fp32 state, no bf16 rounding anywhere), csrc/gru_f32.cu.  It exists to measure
 * the bf16 tensor-core path against (SURVEY.md section 7), not to be fast.
 *   barrier: ndir u32 words (zeroed by the call).  Constraints: H % 4 == 0, Bp <= 128,
 *   H/8 <= number of SMs. */
int sb_gru_fwd_f32(const float* gi, const float* whh_f32, const float* bhh, float* y,
                   unsigned int* barrier, int T, int Bp, int H, int ndir, void* stream);

/* Backward through the recurrence.
 *   dy     [T*Bp][ndir*H] f32  gradient w.r.t. y
 *   whh    [ndir][3H][H] bf16  recurrent weights as stored (the same operand sb_gru_fwd takes;
 *          the kernel transposes its slice while staging it into shared memory)
 *   dgi    [T*Bp][ndir*3H] bf16 (out) gradient w.r.t. gi  -> dX = dgi * W_ih, dW_ih, dW_hh (r,z)
 *   dghn   [T*Bp][ndir*H] bf16 (out) r * dn_pre            -> dW_hh (n rows)
 *          (the weight gradients contract these token-major operands directly with
 *           SB_GEMM_A_MN | SB_GEMM_B_MN; no transposed copies exist)
 *   dbih, dbhh [ndir*3H] f32 accumulated (+=)
 *   workspace  >= sb_gru_bwd_workspace_size bytes, 1024-byte aligned (zeroed by the call itself)
 */
int sb_gru_bwd_workspace_size(int Bp, int H, int ndir, size_t* bytes);
int sb_gru_bwd(const float* dy, const float* y, const float* gates, const void* whh_bf16,
               void* dgi_bf16, void* dghn_bf16, float* dbih, float* dbhh, void* workspace,
               size_t workspace_bytes, int T, int Bp, int H, int ndir, void* stream);

/* ---------------------------------------------------------------------------------------
 * CTC prefix beam search, one CTA per utterance.
 * Replaces: speech.models.ctc_decoder.decode(probs, beam_size, blank)
 *           (speech/models/ctc_decoder.py:38-113; called per utterance by CTC.infer,
 *            speech/models/ctc_model.py:55-60).
 *   logp        (B, T, S) float32 LOG-probabilities (the reference takes np.log of its input
 *               first, ctc_decoder.py:52)
 *   lens        (B) int32 frames to decode per utterance (<= T)
 *   out_labels  (B, T) int32, out_lens (B) int32: best prefix of each utterance
 *   out_scores  (B) float64: negative log-likelihood of that prefix (ctc_decoder.py:112-113)
 * beam_size <= 32.  Lattice arithmetic is float64, ties are broken like the reference's
 * stable sort over dict insertion order.
 * ------------------------------------------------------------------------------------- */
int sb_ctc_prefix_beam_workspace_size(int B, int T, int beam_size, size_t* bytes);
int sb_ctc_prefix_beam(const float* logp, const int* lens, int B, int T, int S, int beam_size,
                       int blank, int* out_labels, int* out_lens, double* out_scores,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Conv2d(+ReLU) front-end as im2col + sb_gemm_bf16_tn.
 * Replaces: the cuDNN convolutions behind nn.Conv2d in Model.encode
 *           (speech/models/model.py:19-29,60-71; valid conv, kernel (kh,kw), stride s both dims).
 * Activations are pixel-major channels-last f32 P[(b*To+t)*Fo+f][c] (= the GEMM's C matrix, ReLU
 * applied on read); the im2col matrix is A[m][(i*kw+j)*Ci+ci] bf16 with K padded to Kp.
 *   sb_conv_im2col       src P (or the (B,T,F) input with Ci=1) -> A
 *   sb_conv_relu_to_bct  C of the last layer -> (B, To, Co*Fo) f32 with ReLU (model.py:66-71)
 *   sb_conv_dtop         dY (B,To,Co*Fo) * (C>0) -> dC bf16 [M][Co]; db[c] += column sums
 *   sb_conv_col2im_relu  dA f32 [M][ldA] -> dC of the layer below (gather, masked by Pprev>0)
 * ------------------------------------------------------------------------------------- */
/* `mask_u8` (may be NULL): dropout keep-bytes (1 keep, 0 drop) of the activations involved, same
 * pixel-major channels-last layout as those activations; kept values are multiplied by `mscale`
 * = 1/(1-p) (nn.Dropout after ReLU, model.py:25-26). */
int sb_conv_im2col(const float* src, const void* mask_u8, float mscale, void* dst_bf16, int B,
                   int Ti, int Fi, int Ci, int kh, int kw, int stride, int Kp, int relu,
                   void* stream);
int sb_conv_relu_to_bct(const float* C, const void* mask_u8, float mscale, float* out, int B,
                        int To, int Fo, int Co, void* stream);
int sb_conv_dtop(const float* dY, const float* C, const void* mask_u8, float mscale,
                 void* dC_bf16, float* db, int B, int To, int Fo, int Co, void* stream);
int sb_conv_col2im_relu(const float* dA, long long ldA, const float* Pprev,
                        const void* maskprev_u8, float mscale, void* dCprev_bf16, float* db, int B,
                        int Ti, int Fi, int Ci, int kh, int kw, int stride, void* stream);

/* ---------------------------------------------------------------------------------------
 * Tail of the training step over flat fp32 buffers.
 * Replaces: nn.utils.clip_grad_norm(model.parameters(), 200) + torch.optim.SGD.step()
 *           (train.py:32-35, 95-97).
 *   sb_sumsq          out[0] = sum(g^2), one pass over the gradient; per-CTA partials combined in
 *                     a fixed order (bit-reproducible: data-parallel replicas stay identical);
 *                     workspace: sb_sumsq_workspace_size bytes, zeroed once by the caller
 *   sb_sgd_clip_step  c = min(1, max_norm/(sqrt(sumsq)+1e-6)); [m = momentum*m + c*g]; p -= lr*(m|c*g)
 *                     the clip coefficient is read from device memory (no host sync);
 *                     params_bf16 (may be NULL): bf16 copy of the updated parameters, the
 *                     tensor-core operands of the next step (no per-step cast kernels)
 * ------------------------------------------------------------------------------------- */
int sb_sumsq_workspace_size(size_t* bytes);
int sb_sumsq(const float* g, long long n, float* out, void* workspace, void* stream);
int sb_sgd_clip_step(float* params, const float* grads, float* momentum_buf, void* params_bf16,
                     long long n, const float* sumsq, float lr, float momentum, float max_norm,
                     void* stream);

/* ---------------------------------------------------------------------------------------
 * Attention decoder step of the sequence-to-sequence model (csrc/s2s.cu), fp32.
 * Replaces: the per-token chain nn.Embedding + nn.GRUCell + NNAttention (Conv1d, broadcast add,
 *           ReLU, Linear, softmax, weighted sum) + LinearND of Seq2Seq.decode / decode_step
 *           (speech/models/seq2seq.py:78-137, 344-360) and the host loops of infer (:145-178) and
 *           beam_search (:180-227).
 *   sb_s2s_cell_fwd   ix = emb[tok[b*tok_stride]] + sx_prev (NULL at the first step);
 *                     hx = GRUCell(ix, hx_prev); optionally saves ix and the gates (r, z, n, hn)
 *   sb_s2s_attn_fwd   attention of every row over eh (eh_bcast: all rows attend over utterance
 *                     0 - beam search), sx (B,H) / ax (B,T); with fc_w: logits = fc(hx + sx) written
 *                     at logits[b*logit_stride + c], optional log-softmax, arg-max, greedy history
 *                     and end-token count; `done` (device int, may be NULL): != 0 -> no-op
 *   sb_attn_step      the attention alone (NNAttention.forward on the decode path)
 *   sb_s2s_dout       backward of the output projection for all (step, utterance) rows at once:
 *                     d_o = dlogits W_fc, o = hx + sx (operand of the time-batched d W_fc)
 *   sb_s2s_attn_bwd / sb_s2s_cell_bwd   gradients of one step (see csrc/s2s.cu)
 *   sb_s2s_check_done greedy stop rule: every row emitted end_tok in the same step
 *   sb_s2s_beam_*     device-side beam bookkeeping with the reference's stable-sort tie order
 * Layouts that differ from the reference's parameters (transposed once per call by the host
 * mirror): conv_wT (Kc, H) = NNAttention.conv.weight (H, 1, Kc) transposed; w_ihT / w_hhT (H, 3H)
 * = GRUCell weights transposed (backward only).  g_conv_wT is (B, ceil(T/24), Kc, H): one slot
 * per CTA, accumulated over the steps, to be summed over its two leading dims by the caller.
 * workspace: >= sb_s2s_workspace_size(B, T, H) bytes, its first 4*B bytes ZERO before the first
 * call (ticket counters; the kernels leave them zero); one workspace serves all steps.
 * Constraints: H % 4 == 0 (attention backward: H <= 1664, its shared-memory tile is 33 H floats),
 * conv kernel width odd and <= 15, T <= 6144, beam <= 32.
 * ------------------------------------------------------------------------------------- */
int sb_s2s_workspace_size(int B, int T, int H, size_t* bytes);
int sb_attn_step(const float* eh, const float* dhx, const float* ax_prev, const float* conv_wT,
                 const float* conv_b, const float* lin_w, float lin_b, int log_t, int B, int T,
                 int H, int Kc, float* sx, float* ax, void* workspace, size_t workspace_bytes,
                 void* stream);
int sb_s2s_cell_fwd(const float* emb, const int* tok, int tok_stride, const float* sx_prev,
                    const float* hx_prev, const float* w_ih, const float* w_hh, const float* b_ih,
                    const float* b_hh, float* hx, float* ix_save, float* gates_save,
                    const int* done, int B, int H, void* stream);
int sb_s2s_attn_fwd(const float* eh, int eh_bcast, const float* hx, const float* ax_prev,
                    const float* conv_wT, const float* conv_b, const float* lin_w, float lin_b,
                    int log_t, int B, int T, int H, int Kc, float* sx, float* ax,
                    const float* fc_w, const float* fc_b, int C, float* logits,
                    long long logit_stride, float* logp, int* argmax, int* history,
                    int hist_stride, int hist_col, int* end_count, int end_tok, const int* done,
                    void* workspace, size_t workspace_bytes, void* stream);
int sb_s2s_dout(const float* dlogits, const float* fc_w, const float* hx, const float* sx,
                float* d_o, float* o_all, long long rows, int C, int H, void* stream);
int sb_s2s_attn_bwd(const float* eh, const float* hx, const float* hx_prev, const float* ax_prev,
                    const float* ax, const float* conv_wT, const float* conv_b,
                    const float* lin_w, const float* d_o, const float* d_ix_next,
                    const float* d_ax_next, const float* d_hx_next, const float* gates,
                    float* d_eh, float* d_ax_prev, float* d_gi, float* d_gh, float* d_hx_direct,
                    float* g_conv_wT, float* g_conv_b, float* g_lin_w, float* g_lin_b, int log_t,
                    int B, int T, int H, int Kc, void* workspace, size_t workspace_bytes,
                    void* stream);
int sb_s2s_cell_bwd(const float* d_gi, const float* d_gh, const float* d_hx_direct,
                    const float* w_ihT, const float* w_hhT, float* d_ix, float* d_hx_prev, int B,
                    int H, void* stream);
int sb_s2s_check_done(const int* end_count, int B, int* done, int* nsteps, int step1, void* stream);
int sb_s2s_beam_state_size(size_t* bytes);
int sb_s2s_beam_init(void* state, int* nodes, int* tok_next, int start_tok, void* stream);
int sb_s2s_beam_select(const float* logp, void* state, double* c_scores, int* nodes,
                       int* parent_row, int* tok_next, int* out_tokens, int K, int C, int end_tok,
                       int step, int max_len, int node_cap, int c_cap, void* stream);
int sb_s2s_beam_gather(const float* hx_in, const float* sx_in, const float* ax_in, float* hx_out,
                       float* sx_out, float* ax_out, const int* parent_row, const void* state,
                       int K, int H, int T, void* stream);

/* Beam expand/prune of Seq2Seq.beam_search (speech/models/seq2seq.py:200-212): indices and values
 * of the k best of n float64 scores, ordered by (score descending, index ascending) - the order of
 * the reference's stable sort over (beam, vocab) candidates. */
int sb_beam_topk(const double* scores, int n, int k, int* out_idx, double* out_val, void* stream);

/* ---------------------------------------------------------------------------------------
 * RNN-Transducer loss + gradient w.r.t. the log-probabilities.
 * Replaces: transducer.functions.transducer.TransducerLoss()(log_probs, labels, x_lens, y_lens)
 *           (libs/transducer, un-vendored, Makefile:10-12; call site
 *            speech/models/transducer_model.py:46-52).
 *   log_probs (B, T, U1, V) float32 log-softmax over V (U1 = max label length + 1)
 *   grads     same shape, out (zero-filled here, then the 2 non-zero entries per cell); may be NULL
 *   labels    flat int32; label_offsets exclusive prefix sum; label_lens (B); act_lens (B)
 *   blank     blank class index (reference: V-1, transducer_model.py:28)
 *   costs     (B) float32 out
 * ------------------------------------------------------------------------------------- */
int sb_rnnt_workspace_size(int B, int T, int U1, size_t* bytes);
int sb_rnnt_fwd_bwd(const float* log_probs, float* grads, const int* labels,
                    const int* label_offsets, const int* label_lens, const int* act_lens, int B,
                    int T, int U1, int V, int blank, float* costs, void* workspace,
                    size_t workspace_bytes, void* stream);

/* Compact-lattice form of the same loss: `lat` / `garc` are (T, B, U1, 2), TIME-major nodes
 * n = (t*B + b)*U1 + u, = {log p(blank), log p(label of arc u -> u+1)} per node (what
 * sb_rnnt_joint_fwd writes) and the gradients w.r.t. them. */
int sb_rnnt_fwd_bwd_compact(const float* lat, float* garc, const int* labels,
                            const int* label_offsets, const int* label_lens, const int* act_lens,
                            int B, int T, int U1, int blank, float* costs, void* workspace,
                            size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Fused RNN-T joint network: relu(fx[b,t,:] + fy[b,u,:]) -> fc2 -> log-softmax per lattice node,
 * the (B, T', U+1, H) intermediate never exists (it lives as 16 KB operand tiles in shared memory).
 * Replaces: the broadcast add + ReLU + LinearND + log_softmax of Transducer.decode,
 *           speech/models/transducer_model.py:71-76 (fc1 shared by both streams, :73).
 *   fx [B*T][H] f32 = fc1(encoder states), fy [B*U1][H] f32 = fc1(prediction network) (biases in)
 *   w2 [V1][H] bf16, b2 [V1] f32: fc2;  ymat [B][U1-1] int32 end-padded labels
 *   node order of lat / garc / dlogits: TIME-major, n = (t*B + b)*U1 + u (frames t0..t0+Tc-1
 *   are one contiguous slab of rows)
 *   sb_rnnt_joint_fwd:      lat [nodes][2] (out), lp_full (B, T, U1, V1) batch-first (out, may be
 *                           NULL: only `infer` needs every class)
 *   sb_rnnt_joint_dlogits:  backward recompute pass: garc [nodes][2] (gradient w.r.t. lat) ->
 *                           dlogits [nodes][NV] bf16 (NV = 32 if V1 <= 32 else 64), db2 [V1] +=
 *   sb_rnnt_joint_build_slab / _reduce_slab: the hidden activations of Tc <= 8 frames
 *                           (z [B*Tc*U1][H] bf16) for the weight-gradient GEMMs, and the masked
 *                           reduction of dz [B*Tc*U1][H] f32 into dfx (=) and dfy (+=)
 * Constraints: H % 8 == 0, V1 <= 64.
 * ------------------------------------------------------------------------------------- */
int sb_rnnt_joint_fwd(const float* fx, const float* fy, const void* w2_bf16, const float* b2,
                      const int* ymat, float* lat, float* lp_full, int B, int T, int U1, int H,
                      int V1, int blank, void* stream);
int sb_rnnt_joint_dlogits(const float* fx, const float* fy, const void* w2_bf16, const float* b2,
                          const int* ymat, const float* garc, void* dlogits_bf16, float* db2, int B,
                          int T, int U1, int H, int V1, int blank, void* stream);
int sb_rnnt_joint_build_slab(const float* fx, const float* fy, void* z_bf16, int B, int T, int U1,
                             int H, int t0, int Tc, void* stream);
int sb_rnnt_joint_reduce_slab(const float* dz, const void* z_bf16, float* dfx, float* dfy, int B,
                              int T, int U1, int H, int t0, int Tc, void* stream);

/* ---------------------------------------------------------------------------------------
 * Transducer beam search over a precomputed (teacher-forced) lattice, one CTA per utterance.
 * Replaces: transducer.decoders.decode_static(lp, beam_size, blank) of the un-vendored
 *           awni/transducer, called per utterance on a host array at
 *           speech/models/transducer_model.py:92-101.
 *   lp       (B, T, U1, V) f32 log-probabilities (device)
 *   tlens    (B) frames searched per utterance, ulens (B) lattice rows (labels + 1)
 *   out_labels (B, U1) int32, out_lens (B), out_scores (B) f64 log-probability of the best
 *   workspace >= sb_rnnt_decode_static_workspace_size bytes;  beam_size <= 32
 * ------------------------------------------------------------------------------------- */
int sb_rnnt_decode_static_workspace_size(int B, int T, int U1, int beam_size, size_t* bytes);
int sb_rnnt_decode_static(const float* lp, const int* tlens, const int* ulens, int B, int T, int U1,
                          int V, int beam_size, int blank, int* out_labels, int* out_lens,
                          double* out_scores, void* workspace, size_t workspace_bytes,
                          void* stream);

/* ---------------------------------------------------------------------------------------------
 * Scoring (SURVEY.md section 8f rank 4), HOST function: Levenshtein distance of two int32 token
 * sequences; replaces `editdistance.eval` in speech/utils/score.py:15-16.  Returns -1 on invalid
 * arguments. */
long long sb_edit_distance(const int* a, long long na, const int* b, long long nb);

/* ---------------------------------------------------------------------------------------------
 * Featuriser (SURVEY.md section 8f rank 2).  Replaces speech/loader.py:152-166 `log_specgram`
 * (scipy.signal.spectrogram, periodic Hann window, one-sided density PSD, no detrend / padding,
 * then log(float32(PSD) + eps)) and the normalisation of loader.py:65-67 `(x - mean) / std`.
 *   pcm        int16 samples of all utterances, concatenated (device)
 *   offsets    [B] index of each utterance's first sample in pcm (device, int64)
 *   n_samples  [B] samples per utterance (device, int32)
 *   nperseg    window length in samples (<= 1024), step = nperseg - noverlap
 *   scale      1 / (sample_rate * sum(window^2)), computed by the caller in float64
 *   mean, stdev [nperseg/2+1] per-bin statistics (device, float32) or NULL for the raw log PSD
 *   out        [B][max_frames][nperseg/2+1] float32; frames past an utterance's end are set to 0
 *              (the zero padding of model.py:135-141)
 * Frames per utterance: (n_samples - noverlap) / step if n_samples >= nperseg, else 0. */
int sb_log_specgram(const short* pcm, const long long* offsets, const int* n_samples, int B,
                    int nperseg, int step, double scale, float eps, const float* mean,
                    const float* stdev, float* out, int max_frames, void* stream);

/* Developer hook (not part of the drop-in surface): device buffer of >= 64*16 uint64 receiving a
 * globaltimer timeline of CTA 0 for the next sb_gru_fwd launches; NULL disables. */
int sb_debug_gru_timeline(void* dev_buffer);
/* Developer hook, query only: with query = 0, returns the thread-block-cluster size the last
 * sb_gru_fwd / sb_gru_bwd launch used (0 before the first one); any other argument returns -1. */
int sb_debug_gru_cluster(int query);

#ifdef __cplusplus
}
#endif
#endif /* SPEECH_B200_H_ */
