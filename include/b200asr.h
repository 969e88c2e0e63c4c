/* libb200asr.so - C ABI of the B200-native ASR train-step kernels (sm_100a).
 *
 * The reference (Alexander-H-Liu/End-to-end-ASR-Pytorch) is 100% Python and has no FFI of its own: every
 * "kernel" is a stock torch / torchaudio call.  Each entry point below therefore cites the reference CALL SITE
 * (file:line under /root/reference, or kaldi.py = torchaudio/compliance/kaldi.py) whose arithmetic it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless stated otherwise; tensors are contiguous row-major fp32,
 *     indices / lengths are int64 ("long long") where the reference passes LongTensors, int32 otherwise;
 *   - the library never allocates, frees or retains device memory: the caller owns inputs, outputs and the
 *     workspaces whose sizes the *_workspace_bytes() helpers return;
 *   - all work is enqueued on `stream` (a cudaStream_t) and the call returns without synchronising;
 *   - return value: 0 = ok, <0 = error (-1 invalid argument, -2 CUDA failure); the message is available
 *     from b200asr_last_error() (thread local).  There is no CPU fallback.
 */
#ifndef B200ASR_H
#define B200ASR_H

#include <stddef.h>

#define B200ASR_VERSION 100

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define B200ASR_API __attribute__((visibility("default")))
#else
#define B200ASR_API
#endif

typedef void* b200asr_stream; /* cudaStream_t */

B200ASR_API int b200asr_version(void);
B200ASR_API const char* b200asr_last_error(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
B200ASR_API unsigned long long b200asr_launch_count(void);
B200ASR_API void b200asr_launch_count_reset(void);
B200ASR_API int b200asr_device_sm_count(void);

/* ---- K1: fused STFT + mel + log -----------------------------------------------------------------------
 * replaces src/audio.py:104-108 -> kaldi.py:514-646 (fbank), :44-83 (framing), :154-217 (dc / pre-emphasis /
 * window).  wave [B, n_max] (zero padded), wave_len [B] samples.  window [win_size] and the sparse mel
 * filters (filter i covers FFT bins mel_start[i] .. +mel_count[i], weights at mel_w[mel_off[i] ..]) are
 * caller-built tables.  fbank [B, t_max, n_mel] (frames >= n_frames[b] are zeroed), n_frames [B] (int32 out)
 * = 1 + (len - win_size) / win_shift (snip_edges=True).  n_fft must be 512.                               */
B200ASR_API int b200asr_fbank_fwd(const float* wave, const int* wave_len, int B, int n_max, int win_size, int win_shift,
                      int n_fft, float preemph, int remove_dc, const float* window, int n_mel,
                      const int* mel_start, const int* mel_count, const int* mel_off, const float* mel_w,
                      int mel_w_total, int use_log, float log_floor, float* fbank, int t_max, int* n_frames,
                      b200asr_stream stream);
/* same kernel fed with 16-bit PCM [B, n_max] (what the corpus files hold, src/data.py:14-43 -> torchaudio.load): the
 * int16 -> fp32 conversion (sample / 32768) happens on the fly, so the host-to-device copy is half as large */
B200ASR_API int b200asr_fbank_fwd_pcm16(const short* pcm, const int* wave_len, int B, int n_max, int win_size, int win_shift,
                      int n_fft, float preemph, int remove_dc, const float* window, int n_mel,
                      const int* mel_start, const int* mel_count, const int* mel_off, const float* mel_w,
                      int mel_w_total, int use_log, float log_floor, float* fbank, int t_max, int* n_frames,
                      b200asr_stream stream);

/* ---- K2+K3: delta / delta-delta + per-utterance CMVN + channel-major interleave ---------------------------
 * replaces src/audio.py:51-54,57-77 (Delta), :25-27 (CMVN, unbiased std, eps added to std), :85-89
 * (Postprocess).  feat [B, t_max, n_mel*(delta_order+1)], rows >= n_frames[b] are zero (pad_sequence,
 * src/data.py:39).                                                                                          */
B200ASR_API size_t b200asr_delta_cmvn_workspace_bytes(int B, int t_max, int n_mel, int delta_order);
B200ASR_API int b200asr_delta_cmvn_fwd(const float* fbank, const int* n_frames, int B, int t_max, int n_mel,
                                       int delta_order, int delta_window, int apply_cmvn, float cmvn_eps,
                                       float* feat, void* workspace, size_t workspace_bytes, b200asr_stream stream);

/* ---- K9: log-softmax over the vocabulary (src/asr.py:96) -------------------------------------------------
 * log_probs may alias logits.  lse [n_rows] and argmax [n_rows] (int64; util.py:117-118 / test_asr.py:116-118)
 * are optional (NULL); log_probs may be NULL when lse is given (statistics only, see b200asr_ctc_fwd_bwd_logits). */
B200ASR_API int b200asr_log_softmax_fwd(const float* logits, float* log_probs, float* lse, long long* argmax,
                            long long n_rows, int V, b200asr_stream stream);
B200ASR_API int b200asr_log_softmax_bwd(const float* log_probs, const float* grad_out, float* grad_in, long long n_rows,
                            int V, b200asr_stream stream);

/* ---- K10: CTC loss forward + backward in one call ---------------------------------------------------------
 * replaces torch.nn.CTCLoss(blank=0, zero_infinity=False) at bin/train_asr.py:49,123-124 (ATen _ctc_loss +
 * _ctc_loss_backward).  log_probs element (b,t,c) lives at log_probs[b*stride_b + t*stride_t + c]; targets
 * [B, L_max] zero padded int64; input_lengths / target_lengths [B] int64.  nll [B] out (per-utterance negative
 * log likelihood, +inf when infeasible).  If grad != NULL it receives, with the same strides as log_probs,
 * grad_scale[b] * (exp(lp) - exp(log sum_{s: l'_s = c} alpha_t(s) beta_t(s) + nll - lp)) for t < input_length
 * and 0 after it - ATen's convention (SURVEY.md F9).  grad_scale may be NULL (= 1).                         */
B200ASR_API size_t b200asr_ctc_workspace_bytes(int B, int T, int L_max);
B200ASR_API int b200asr_ctc_fwd_bwd(const float* log_probs, long long stride_b, long long stride_t, const long long* targets,
                        const long long* input_lengths, const long long* target_lengths, int B, int T, int V,
                        int L_max, int blank, float* nll, const float* grad_scale, float* grad, void* workspace,
                        size_t workspace_bytes, b200asr_stream stream);
/* The gradient half alone, for callers that learn the upstream scale only in their backward pass (autograd): run
 * b200asr_ctc_fwd_bwd with grad = NULL in the forward (nll + the alpha/beta lattices stay in `workspace`), then this
 * with the SAME workspace.  `upstream` (device scalar, may be NULL) multiplies every element, so no separate scaling
 * pass over the [T,B,V] gradient is needed.  Out-of-range labels are clamped into [0,V) (torch raises on them). */
B200ASR_API int b200asr_ctc_grad(const float* log_probs, long long stride_b, long long stride_t, const long long* targets,
                     const long long* input_lengths, const long long* target_lengths, int B, int T, int V,
                     int L_max, int blank, const float* nll, const float* grad_scale, const float* upstream,
                     float* grad, void* workspace, size_t workspace_bytes, b200asr_stream stream);

/* The CTC head fused into the loss (src/asr.py:96 + bin/train_asr.py:123-124 in one pass structure): the same two
 * calls on LOGITS plus the per-row log-sum-exp  row_lse[b * T + t]  (b200asr_log_softmax_fwd with log_probs = NULL
 * writes only lse + argmax).  log-prob(b,t,c) = logits[...] - row_lse[b*T + t] is formed on the fly, the V-wide log-prob
 * tensor is never written or re-read, and `grad` IS the logit gradient (exp(x - lse) - occupancy has zero class sum,
 * SURVEY.md F9):  12*T*V bytes per utterance (read logits twice, write the gradient once) instead of 28*T*V.      */
B200ASR_API int b200asr_ctc_fwd_bwd_logits(const float* logits, const float* row_lse, long long stride_b, long long stride_t,
                               const long long* targets, const long long* input_lengths,
                               const long long* target_lengths, int B, int T, int V, int L_max, int blank, float* nll,
                               const float* grad_scale, float* grad, void* workspace, size_t workspace_bytes,
                               b200asr_stream stream);
B200ASR_API int b200asr_ctc_grad_logits(const float* logits, const float* row_lse, long long stride_b, long long stride_t,
                            const long long* targets, const long long* input_lengths, const long long* target_lengths,
                            int B, int T, int V, int L_max, int blank, const float* nll, const float* grad_scale,
                            const float* upstream, float* grad, void* workspace, size_t workspace_bytes,
                            b200asr_stream stream);

/* ---- SURVEY 8(f) rank 3: CTC prefix scoring (joint CTC/attention beam search) ---------------------------------
 * replaces CTCPrefixScore.cheap_compute (src/ctc.py:81-116), called from src/decode.py:129-131 once per hypothesis
 * and step on the host.  Scores N hypotheses x C candidate tokens in one launch.
 *   log_probs  [T, V]      CTC log-probs of the utterance          r_prev   [N, T, 2]  state of each prefix
 *   last_char  [N], prefix_len [N] (int32)                         candidates [N, C] (int32, ids in [0,V))
 *   psi [N, C] out: log P(prefix + c, ...)                         r_out [N, C, T, 2] out: state of prefix + c
 * float32, the reference's finite log-zero (-1e8), numpy.logaddexp formula.  Out-of-range ids are the caller's bug. */
B200ASR_API int b200asr_ctc_prefix_score(const float* log_probs, int T, int V, const float* r_prev, const int* last_char,
                             const int* prefix_len, const int* candidates, int N, int C, int blank, int eos,
                             float* psi, float* r_out, b200asr_stream stream);

/* ---- K7/K8: persistent (Bi)LSTM recurrence -----------------------------------------------------------------
 * replaces the time loop inside torch.nn.LSTM as used by src/module.py:112-113,129-132 (one layer,
 * batch_first, zero initial state, run over the padded frames).  ndir = 1 or 2 (direction 1 = reverse time).
 *   gates  [ndir, B, T, H, 4]  in : input projection x.W_ih^T + b_ih + b_hh, gate-interleaved (i,f,g,o minor)
 *                              out: the activated gates (stash for the backward pass)
 *   w_hh   [ndir, 4H, H]       PyTorch layout (weight_hh_l0 [, weight_hh_l0_reverse])
 *   cstate [ndir, B, T, H]     out: cell state after every step (stash)
 *   out    [B, T, ndir*H]      out: hidden states (the layer output)
 * backward: gates in = stash, out = d(loss)/d(pre-activation) in the same layout; dout [B, T, ndir*H].
 * H must be a multiple of 16; the (unit-block, batch-block) decomposition must fit the SM count
 * (b200asr_bilstm_plan reports it).  Launched cooperatively: all CTAs are co-resident.                       */
B200ASR_API size_t b200asr_bilstm_workspace_bytes(int B, int T, int H, int ndir);
B200ASR_API int b200asr_bilstm_plan(int B, int H, int ndir, int* unit_block, int* batch_block, int* n_ctas);
/* 1 when the step GEMMs of this shape run on the tensor cores (3xTF32 mma), 0 for the packed-fp32-FMA kernels,
 * -1 when the shape has no decomposition */
B200ASR_API int b200asr_bilstm_uses_tensor_cores(int B, int H, int ndir);
/* 1 when the forward recurrence of this shape runs on the 5th-generation tensor cores (tcgen05.mma kind::f16 with
 * fp32 accumulators in TMEM and the fp16 hi/lo "2 x 2 block" split product, csrc/lstm_umma.cu), else 0 */
B200ASR_API int b200asr_bilstm_uses_tcgen05(int B, int H, int ndir);
B200ASR_API int b200asr_bilstm_fwd(float* gates, const float* w_hh, float* cstate, float* out, int B, int T, int H, int ndir,
                       void* workspace, size_t workspace_bytes, b200asr_stream stream);
B200ASR_API int b200asr_bilstm_bwd(float* gates, const float* w_hh, const float* cstate, const float* dout, int B, int T,
                       int H, int ndir, void* workspace, size_t workspace_bytes, b200asr_stream stream);


/* ---- K13: one LSTM cell step (decoder, src/asr.py:214-221) -------------------------------------------------
 * preact [B, 4H] gate-major (i,f,g,o) = x.W_ih^T + h.W_hh^T + biases; gates [B,4H] activated (stash).        */
B200ASR_API int b200asr_lstm_cell_fwd(const float* preact, const float* c_prev, float* gates, float* c, float* h, int B,
                          int H, b200asr_stream stream);
B200ASR_API int b200asr_lstm_cell_bwd(const float* gates, const float* c_prev, const float* c, const float* dh,
                          const float* dc_next /* may be NULL */, float* dpreact, float* dc_prev, int B, int H,
                          b200asr_stream stream);

/* ---- K12: location-aware attention step, forward and backward, one launch each ----------------------------------
 * replaces src/module.py:234-258 (LocationAwareAttention.forward) + :189-195 (_attend), single head:
 * Conv1d(1->K, 2R+1, pad R, no bias) over prev_att -> Linear(K->D, no bias) -> tanh -> energy = Linear(D->1)(tanh(key +
 * q + loc)) / temperature -> masked softmax over t < enc_len[b] -> context = attn . value.
 *   q [B,D] (already tanh(proj_q(h))), key [B,T,D] (tanh(proj_k(enc))), value [B,T,E], prev_att [B,T], enc_len [B] i64,
 *   w_conv [K,2R+1], w_proj [D,K], w_energy [D], b_energy [1]  ->  attn [B,T], ctx [B,E].
 * backward: dctx [B,E], dattn [B,T] or NULL -> dq_part [B,CS,D] (sum over CS = dq), dkey [B,T,D], dvalue [B,T,E],
 * dprev [B,T], wpart [B*CS, P] with P = D*K + K*(2R+1) + D + 1 laid out (d w_proj | d w_conv | d w_energy | d b_energy);
 * the caller sums wpart over its first axis.  CS = b200asr_locattn_cluster_size(T, E) CTAs cooperate per utterance
 * through distributed shared memory.  K <= 16, E % 4 == 0, D <= 512, E / CS <= 1024.                                              */
B200ASR_API int b200asr_locattn_cluster_size(int T, int E);
B200ASR_API size_t b200asr_locattn_wpart_floats(int D, int K, int R);
B200ASR_API int b200asr_locattn_fwd(const float* q, const float* key, const float* value, const float* prev_att,
                                    const long long* enc_len, const float* w_conv, const float* w_proj,
                                    const float* w_energy, const float* b_energy, float temperature, int B, int T,
                                    int D, int E, int K, int R, float* attn, float* ctx, b200asr_stream stream);
B200ASR_API int b200asr_locattn_bwd(const float* q, const float* key, const float* value, const float* prev_att,
                                    const long long* enc_len, const float* w_conv, const float* w_proj,
                                    const float* w_energy, float temperature, const float* attn, const float* dctx,
                                    const float* dattn, int B, int T, int D, int E, int K, int R, float* dq_part,
                                    float* dkey, float* dvalue, float* dprev, float* wpart, b200asr_stream stream);
/* The decode loop's form of the backward (src/asr.py:112-151 calls the attention L times on the SAME key / value):
 * d(key) and the weight-gradient partials are ADDED into per-batch accumulators (zeroed by the caller before the first
 * step) and d(value) is not produced here at all: d(value)[b,t,:] = sum_l attn_l[b,t] * dctx_l[b,:] is formed once after
 * the loop by b200asr_attn_dvalue from the stacked per-step alignments [B,L,T] and context gradients [B,L,E] - instead
 * of a [B,T,E] write per step that autograd then has to re-add L-1 times.                                             */
B200ASR_API int b200asr_locattn_bwd_acc(const float* q, const float* key, const float* value, const float* prev_att,
                                        const long long* enc_len, const float* w_conv, const float* w_proj,
                                        const float* w_energy, float temperature, const float* attn, const float* dctx,
                                        const float* dattn, int B, int T, int D, int E, int K, int R, float* dq_part,
                                        float* dkey_acc, float* dprev, float* wpart_acc, b200asr_stream stream);
B200ASR_API int b200asr_attn_dvalue(const float* attn_steps, const float* dctx_steps, int B, int L, int T, int E,
                                    float* dvalue, int accumulate, b200asr_stream stream);

/* ---- K15: cross-entropy (log-softmax + NLL, ignore_index) forward + logit gradient ----------------------
 * replaces torch.nn.CrossEntropyLoss(ignore_index=0) at bin/train_asr.py:47,127-131.  row_loss [n_rows] =
 * lse(x) - x[target] (0 for ignored rows); dlogits (optional) = grad_scale[0] * (softmax(x) - onehot), zero rows
 * for ignored targets; grad_scale is a DEVICE scalar (e.g. 1 / number of non-ignored rows) or NULL (= 1).     */
B200ASR_API int b200asr_ce_fwd_bwd(const float* logits, const long long* target, long long ignore_index,
                                   long long n_rows, int V, const float* grad_scale, float* row_loss,
                                   float* dlogits, b200asr_stream stream);

/* ---- K17: token embedding (the RNN-LM's nn.Embedding, src/lm.py:17) forward and weight gradient --------------
 * embedding_fwd: out[n, :] = W[ids[n], :] for n < N; W [V, E], out [N, E] row-major; id 0 is an ordinary row.
 * embedding_bwd: dW[v, :] (accumulate ? += : =) sum of dY[n, :] over the n with ids[n] == v.  `sorted_ids` are the ids
 *   sorted ascending with a STABLE sort and `order` the matching permutation (sorted_ids[i] == ids[order[i]]); each
 *   row's sum runs in ascending position without atomics, so results are bit-reproducible.  Without `accumulate`
 *   the rows that receive no id are zeroed.
 * Ids outside [0, V) are never read through: the forward writes a zero row, the backward skips them (the caller is
 * expected to reject them; ops.embedding does).                                                                     */
B200ASR_API int b200asr_embedding_fwd(const long long* ids, long long N, const float* W, long long V, int E, float* out,
                                      b200asr_stream stream);
B200ASR_API int b200asr_embedding_bwd(const long long* sorted_ids, const long long* order, long long N, const float* dY,
                                      long long V, int E, float* dW, int accumulate, b200asr_stream stream);

/* ---- K16: gradient norm, clip and optimizer update on flat buffers (src/solver.py:84-89, src/optim.py) ----
 * grad_norm (device scalar) may be NULL (no clipping, no NaN skip); max_norm <= 0 disables clipping.          */
B200ASR_API size_t b200asr_grad_norm_scratch_bytes(void);
B200ASR_API int b200asr_grad_norm(const float* grad, long long n, float* norm_out, void* scratch, b200asr_stream stream);
B200ASR_API int b200asr_adadelta_step(float* param, const float* grad, float* square_avg, float* acc_delta, long long n,
                          float lr, float rho, float eps, float weight_decay, const float* grad_norm,
                          float max_norm, b200asr_stream stream);
B200ASR_API int b200asr_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                      float beta1, float beta2, float eps, float weight_decay, int step, const float* grad_norm,
                      float max_norm, b200asr_stream stream);

/* ---- K6 / K9 / K11: dense  x . W^T (+ bias)  on the tensor cores at fp32-class accuracy ------------------------------
 * replaces the input projection inside nn.LSTM (src/module.py:112-113,131), the CTC head (src/asr.py:29,96) and the
 * proj_k / char_trans / pj Linear layers (src/asr.py:177,220,242-243; src/module.py:123,155) and their input gradients.
 *   C[M,N] (+)= A[M,K] . B[N,K]^T + bias[N]      A, B row-major with K contiguous (16-byte aligned, K % 4 == 0),
 *   C row-major with leading dimension ldc >= N; bias may be NULL; accumulate != 0 adds to the existing C.
 * tcgen05.mma kind::tf32 with error compensation: raw fp32 tiles are the TF32 hi operands (the tensor core truncates),
 * the residual tiles are produced on the fly in shared memory; three products per K block into one TMEM accumulator. */
B200ASR_API int b200asr_gemm3x_supported(int M, int N, int K);
B200ASR_API int b200asr_gemm3x_tn(const float* A, const float* B, const float* bias, float* C, int M, int N, int K, int ldc,
                      int accumulate, b200asr_stream stream);
/* same with an explicit row pitch lda (floats, multiple of 4) of A.  lda < K is allowed: overlapping rows are the im2col
 * view of a strided 1-D convolution over a [time, channels] buffer (CNNExtractor, src/module.py:75-78: kernel 4, stride 2
 * -> K = 4*C, lda = 2*C), so the convolution runs in this kernel without materialising the windows. */
B200ASR_API int b200asr_gemm3x_tn_ld(const float* A, int lda, const float* B, const float* bias, float* C, int M, int N, int K,
                         int ldc, int accumulate, b200asr_stream stream);
/* input gradient  dX = dY . W  (autograd backward of the Linear / LSTM input projection above):
 *   C[M,N] (+)= A[M,K] . B[K,N] + bias[N]       A row-major with K contiguous (pitch lda), B row-major with N contiguous
 * (pitch ldb): the weight matrix is read in place as an MN-major tensor-core operand - no transposed copy. */
B200ASR_API int b200asr_gemm3x_nn(const float* A, int lda, const float* B, int ldb, const float* bias, float* C, int M, int N,
                      int K, int ldc, int accumulate, b200asr_stream stream);
/* weight gradient  dW = dY^T . X  (autograd backward of the same layers; contraction over the batch*time rows):
 *   C[m,n] (+)= sum_{b < batches} sum_{t < T}  A[b][t + a_shift][m] * B[b][t + b_shift][n]
 * element (b, t, c) of an operand lives at ptr[b * bstride + t * ld + c] (both operands MN-major); rows outside [0, T)
 * read as zero, so  b_shift = -1 / +1  contracts dG[t] with the hidden state of the PREVIOUS step of the forward /
 * reverse direction (dW_hh of nn.LSTM) straight from the layer output.  permute_rows != 0 writes row m of the result
 * to row (m % 4) * (M / 4) + m / 4: from the kernels' unit-major gate order back to PyTorch's gate-major rows.
 * Small M x N with a long contraction is cut into split-K slices over all SMs (partials in `workspace`, summed in a
 * fixed order by a second launch); workspace may be NULL (no split).                                              */
B200ASR_API size_t b200asr_gemm3x_workspace_bytes(int M, int N);
/* the tn / nn forms with a split-K workspace (b200asr_gemm3x_workspace_bytes(M, N)): skinny products - the decoder's
 * per-step  [B, in] . W^T  with B = 64 rows (src/asr.py:214-221) - are cut along K over all SMs, partial tiles summed in
 * a fixed order by a second launch (bias / accumulate applied there).                                              */
B200ASR_API int b200asr_gemm3x_tn_ws(const float* A, int lda, const float* B, const float* bias, float* C, int M, int N, int K,
                         int ldc, int accumulate, void* workspace, size_t workspace_bytes, b200asr_stream stream);
B200ASR_API int b200asr_gemm3x_nn_ws(const float* A, int lda, const float* B, int ldb, const float* bias, float* C, int M,
                         int N, int K, int ldc, int accumulate, void* workspace, size_t workspace_bytes,
                         b200asr_stream stream);
B200ASR_API int b200asr_gemm3x_nt(const float* A, long long lda, long long a_bstride, int a_shift, const float* B,
                      long long ldb, long long b_bstride, int b_shift, float* C, int M, int N, int T, int batches,
                      int ldc, int accumulate, int permute_rows, void* workspace, size_t workspace_bytes,
                      b200asr_stream stream);

/* the tn / nn forms with a PRE-SPLIT B operand: B_lo = B - trunc_tf32(B) (b200asr_tf32_residual; same shape and pitch
 * as B) is the weight matrix' residual, computed once per step instead of once per tile by every CTA: its tile arrives
 * by TMA like B's, the in-kernel splitter pass shrinks to the A tile and 8 of the 12 tensor-core products of a K block
 * no longer wait for it.  workspace may be NULL.                                                                    */
B200ASR_API int b200asr_tf32_residual(const float* x, float* lo, long long n, b200asr_stream stream);
B200ASR_API int b200asr_gemm3x_tn_pre(const float* A, int lda, const float* B, const float* B_lo, const float* bias, float* C,
                          int M, int N, int K, int ldc, int accumulate, void* workspace, size_t workspace_bytes,
                          b200asr_stream stream);
B200ASR_API int b200asr_gemm3x_nn_pre(const float* A, int lda, const float* B, const float* B_lo, int ldb, const float* bias,
                          float* C, int M, int N, int K, int ldc, int accumulate, void* workspace,
                          size_t workspace_bytes, b200asr_stream stream);
/* all three forms with BOTH operands pre-split: A_lo = A - trunc_tf32(A) has the shape and pitches of A (an activation
 * or gradient matrix that enters several products of the step - the layer input x: forward projection and dW_ih; the
 * gate gradient dG: dX, dW_ih and dW_hh - so one elementwise pass replaces the per-tile split in each of them).  The
 * kernel then has no splitter pass at all: the 12 products of a K block are issued as soon as the four tiles have
 * landed.  Same residuals and the same 12 products per K block as the other entry points (the issue order of the
 * products differs, so results agree to fp32 rounding, not bit for bit).                                            */
B200ASR_API int b200asr_gemm3x_tn_pre2(const float* A, const float* A_lo, int lda, const float* B, const float* B_lo,
                           const float* bias, float* C, int M, int N, int K, int ldc, int accumulate, void* workspace,
                           size_t workspace_bytes, b200asr_stream stream);
B200ASR_API int b200asr_gemm3x_nn_pre2(const float* A, const float* A_lo, int lda, const float* B, const float* B_lo, int ldb,
                           const float* bias, float* C, int M, int N, int K, int ldc, int accumulate, void* workspace,
                           size_t workspace_bytes, b200asr_stream stream);
B200ASR_API int b200asr_gemm3x_nt_pre(const float* A, const float* A_lo, long long lda, long long a_bstride, int a_shift,
                          const float* B, const float* B_lo, long long ldb, long long b_bstride, int b_shift, float* C,
                          int M, int N, int T, int batches, int ldc, int accumulate, int permute_rows, void* workspace,
                          size_t workspace_bytes, b200asr_stream stream);

/* ---- K6 helper: split fp32 into a TF32-representable high part and the fp32 residual ---------------------------
 * hi = x rounded to TF32, lo = x - hi; used to run the input-projection (src/module.py:131, inside nn.LSTM) and the
 * weight-gradient contractions as three error-compensated TF32 tensor-core GEMMs (3xTF32) at fp32-level accuracy.  */
B200ASR_API int b200asr_split_tf32(const float* x, float* hi, float* lo, long long n, b200asr_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* B200ASR_H */
