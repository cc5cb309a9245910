/* wsae.h — C ABI of libwsae_sm100.so: the B200 (sm_100a) TopK-SAE train-step kernels.
 *
 * The reference (omarkhursheed/whisper-sae) is pure PyTorch and has no FFI; each entry point
 * below cites the reference lines (under /root/reference/src/whisper_sae/) whose arithmetic it
 * replaces.  INTEGRATION.md shows the ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch tensors); the library never
 *     allocates, frees or retains them past the call;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value: 0 ok; <0 argument/shape error (WSAE_E_*); >0 a cudaError_t; >=1000 is
 *     1000 + CUresult from the tensor-map encoder;
 *   - global state: per-device "function attribute set" flags (written once), the WSAE_PDL
 *     environment switch (read once) and - EXPERIMENTS ONLY - the process-wide switches behind the
 *     four wsae_debug_* setters at the end of this header (kernel variant / mode / counter buffer /
 *     cluster size read by wsae_encode_topk and wsae_wgrad_gemm at launch time).  A process that
 *     never calls wsae_debug_* may call every other entry point from different host threads on
 *     different streams/devices; the setters themselves are not thread-safe.
 */
#ifndef WSAE_H_
#define WSAE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WSAE_OK 0
#define WSAE_E_BADARG (-1)
#define WSAE_E_UNSUPPORTED (-2)
#define WSAE_E_NODRIVER (-3)

typedef void* wsae_stream_t; /* cudaStream_t */

/* Library / build identification: returns 100 * major + minor of the ABI (currently 111: + wsae_encode_topk_dense, wsae_encode_dense, wsae_row_step with the fused counters, wsae_graph_launch, wsae_memcpy_async; later
 * additions that change no existing behaviour keep the number: wsae_encode_topk_chunked, and k up to 256 in
 * wsae_decode_backward / _at / _rows_at; the half-precision activation forms wsae_pack_activations_typed,
 * wsae_decode_backward_typed, wsae_row_step_typed and wsae_layernorm_rows_typed, whose dtype 0 is the
 * existing entry point; wsae_splice_pack and wsae_splice_decode).
 *
 * Activation dtype codes (x_dtype / in_dtype / out_dtype): 0 = float32, 1 = bfloat16, 2 = float16.  A
 * bf16 / fp16 activation matrix is converted to fp32 as it is loaded, and everything after the load is
 * the fp32 arithmetic: a half matrix Xh gives bit for bit what its fp32 copy Xh.float() gives.  A form
 * that cannot read the given dtype returns WSAE_E_UNSUPPORTED (it never reinterprets the bytes); an
 * unknown code is WSAE_E_BADARG. */
int wsae_abi_version(void);

/* cudaGraphLaunch(graph_exec, stream) for an instantiated CUDA graph of the calls below (the host mirror
 * captures one train step per batch shape; sae/training.py:161-217 is the step it replaces). */
int wsae_graph_launch(void* graph_exec /* cudaGraphExec_t */, wsae_stream_t stream);

/* cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, stream). */
int wsae_memcpy_async(void* dst, const void* src, size_t bytes, wsae_stream_t stream);

/* ---- K0: operand packing (sae/model.py:108 `x - b_pre`; bias of nn.Linear at :111) ------------
 * Packed row layout: `terms` blocks of dp = round_up(d, 8) bf16 columns (split-bf16 pieces), then
 * a 16-column bias block, zero-padded to Kp = round_up(terms*dp + 16, 64).  terms: 1 = bf16,
 * 3 = ~2^-16, 6 = fp32-grade.  Rows >= B up to Bp are written as zeros; encoder rows >= F up to Fp
 * are zeros with a -inf bias, so their pre-activation is -inf and no TopK selects them.
 * Bp must be a multiple of 128 and Fp a multiple of 256 for wsae_encode_topk. */
int wsae_packed_k(int d, int terms, int* dp_out, int* used_cols_out, int* kp_out);
int wsae_pack_activations(const float* x, const float* b_pre /*nullable*/, int B, int Bp, int d,
                          int terms, void* a_packed /*bf16 [Bp,Kp]*/, wsae_stream_t stream);
/* As wsae_pack_activations, but the matrix is named by a device-resident pointer slot: the kernel
 * reads *x_at when it RUNS, so a captured CUDA graph trains on whichever batch the slot names at
 * replay time, in place (reference: training.py:170 hands `model(batch)` the batch itself, no
 * staging copy).  *x_at: 16-byte aligned, B x d fp32.  terms == 1 and d % 8 == 0 only
 * (WSAE_E_UNSUPPORTED otherwise). */
int wsae_pack_activations_at(const float* const* x_at, const float* b_pre /*nullable*/, int B,
                             int Bp, int d, int terms, void* a_packed /*bf16 [Bp,Kp]*/,
                             wsae_stream_t stream);
/* Slot form with a row-index indirection: batch row r is row (*rows_at)[r] of the matrix *x_at names
 * (*rows_at == NULL: identity; indices are int64, as torch.randperm yields them).  Lets the trainer
 * walk a shuffled epoch over a device-resident activation matrix without materialising each batch
 * (reference: DataLoader(TensorDataset(features), shuffle=True), data/feature_cache.py:169-197). */
int wsae_pack_activations_rows_at(const float* const* x_at, const long long* const* rows_at,
                                  const float* b_pre /*nullable*/, int B, int Bp, int d, int terms,
                                  void* a_packed /*bf16 [Bp,Kp]*/, wsae_stream_t stream);
/* Slot form for any activation dtype: *x_at holds B x d elements of type x_dtype (16-byte aligned);
 * rows_at nullable (and *rows_at == NULL: identity).  terms == 1 and d % 8 == 0 only. */
int wsae_pack_activations_typed(const void* const* x_at, const long long* const* rows_at /*nullable*/,
                                int x_dtype, const float* b_pre /*nullable*/, int B, int Bp, int d, int terms,
                                void* a_packed /*bf16 [Bp,Kp]*/, wsae_stream_t stream);
int wsae_pack_encoder(const float* w_enc /*[F,d]*/, const float* b_enc /*[F] nullable*/, int F,
                      int Fp, int d, int terms, void* w_packed /*bf16 [Fp,Kp]*/,
                      wsae_stream_t stream);

/* ---- K1: encoder GEMM + fused per-row TopK (sae/model.py:111 Linear, :114 torch.topk) ---------
 * pre = A' . W'^T on tcgen05 tensor cores (fp32 accumulate in TMEM); the [B,F] pre-activations
 * are never written.  Emits, per row, the k largest pre-activations (signed, pre-ReLU) and their
 * feature indices, unordered.  Ties at the k-th value resolve to the lowest feature index; NaN is
 * never selected; a row with fewer than k non-NaN pre-activations is padded with (-inf, -1), so every
 * index is in [-1, F).  nsplit > 1 splits F across CTAs (latency at small B); part_* are [B, nsplit_eff*k] scratch
 * (nsplit_eff from wsae_encode_effective_splits) and may be NULL when nsplit == 1.  k <= 64
 * (larger k: wsae_encode_topk_dense or wsae_encode_topk_chunked). */
int wsae_encode_effective_splits(int F, int nsplit);
int wsae_encode_topk(const void* a_packed, const void* w_packed, int B, int Bp, int F, int Fp,
                     int Kp, int k_used_cols, int k, int nsplit, float* part_val,
                     int32_t* part_idx, float* out_val /*[B,k]*/, int32_t* out_idx /*[B,k]*/,
                     wsae_stream_t stream);

/* Small-batch form (the shipped configs/tiny_default.yaml trains on 128-row batches): the same GEMM
 * stores its [B,F] pre-activations to `pre_ws` (B*F floats of scratch, L2 resident at these sizes) and
 * one thread block per row selects the k largest with a radix select - no F-split, no merge.  Same
 * values and tie rule as wsae_encode_topk; output in ascending feature index.  F <= 49152, F % 4 == 0. */
int wsae_encode_topk_dense(const void* a_packed, const void* w_packed, int B, int Bp, int F, int Fp,
                           int Kp, int k_used_cols, int k, float* pre_ws, float* out_val /*[B,k]*/,
                           int32_t* out_idx /*[B,k]*/, wsae_stream_t stream);

/* K1 for k > 64 (the fused epilogue of wsae_encode_topk stops at k = 64): the GEMM and row select of
 * wsae_encode_topk_dense over consecutive chunks of chunk_rows packed rows (a multiple of 128), one
 * library call, at any F.  pre_ws is scratch reused by every chunk (size it to stay in L2: ~32-48 MB):
 * chunk_rows * Fr floats with Fr = round_up(F, 4) when F <= 49152; above that the select runs on
 * nslices = ceil(F / 49152) column slices, whose k candidates each are merged, and pre_ws needs
 * chunk_rows * (Fr + 2 * nslices * k) floats.  Same values and tie rule as wsae_encode_topk_dense
 * (bit-identical to one such call over all B rows where that call runs); output in ascending feature
 * index.  k <= 65535, and ceil(nslices * k / 32) <= 64 (F up to 393216 at k = 256):
 * WSAE_E_UNSUPPORTED otherwise. */
int wsae_encode_topk_chunked(const void* a_packed, const void* w_packed, int B, int Bp, int F, int Fp,
                             int Kp, int k_used_cols, int k, int chunk_rows, float* pre_ws,
                             float* out_val /*[B,k]*/, int32_t* out_idx /*[B,k]*/, wsae_stream_t stream);

/* The GEMM half alone: pre_ws[B, F] = A' x W'^T with the bias (sae/model.py:111), no selection. */
int wsae_encode_dense(const void* a_packed, const void* w_packed, int B, int Bp, int F, int Fp, int Kp,
                      int k_used_cols, float* pre_ws, wsae_stream_t stream);

/* ---- Small-batch row step (sae/model.py:114-116,129,145,148,174-181 + their autograd) -----------
 * One thread block per activation row: TopK of pre[row, :] (written to out_val / out_idx, ascending
 * feature index), relu, sparse decode + residual against `target` (or *target_at, row (*rows_at)[row]
 * when rows_at != NULL), SSE + L0 into stats {double sse; uint64 l0} (caller-zeroed), fired stamps
 * (last_activated[f] = *step_count + 1), dv, and the gradient ACCUMULATIONS (all caller-zeroed, fp32
 * atomics): d_b_enc[F], d_b_dec[d], d_w_enc[F,d] += dv * (x - b_pre), d_w_decT[F,d] += coef*g*relu(v)*resid.
 * With w_enc (fp32 [F,d]) and d_b_pre both given, d_b_pre[d] += coef*g*resid - sum_j dv_j * w_enc[i_j, :]
 * (= db_dec - db_enc . W_enc summed over the rows, the job of wsae_bpre_grad).
 * With ticket (a caller-zeroed uint32) given, the LAST block to finish also does wsae_counters_update_post's
 * job: *step_count += 1, *dead_count = #{f: step - last_activated[f] > dead_threshold}, and {sse, l0, dead,
 * *seq} posted to the pinned host `mailbox` (4 x int64) behind a system-scope fence.
 * resid / dpre_val / any gradient pointer may be NULL.  k <= 32, d even, (F + 2 d) * 4 <= 200 KB.
 * Replaces wsae_encode_topk_dense's selection + wsae_decode_backward + wsae_bucket_by_tile + 2 x
 * wsae_wgrad_gemm for batches of a few hundred rows (the shipped YAML batch is 128). */
int wsae_row_step(const float* pre, const float* target, const float* const* target_at,
                  const long long* const* rows_at, const void* w_decT_bf16, const float* b_dec,
                  const float* b_pre, const float* grad_out, float coef, int B, int d, int F, int k,
                  float* out_val, int32_t* out_idx, void* stats, long long* last_activated,
                  long long* step_count, float* d_b_enc, float* d_b_dec, float* d_w_enc,
                  float* d_w_decT, float* resid, float* dpre_val, const float* w_enc, float* d_b_pre,
                  unsigned int* ticket, long long dead_threshold, long long* dead_count,
                  const long long* seq, long long* mailbox, wsae_stream_t stream);
/* As wsae_row_step, with target / *target_at of element type x_dtype. */
int wsae_row_step_typed(const float* pre, const void* target, const void* const* target_at,
                        const long long* const* rows_at, int x_dtype, const void* w_decT_bf16, const float* b_dec,
                        const float* b_pre, const float* grad_out, float coef, int B, int d, int F, int k,
                        float* out_val, int32_t* out_idx, void* stats, long long* last_activated,
                        long long* step_count, float* d_b_enc, float* d_b_dec, float* d_w_enc,
                        float* d_w_decT, float* resid, float* dpre_val, const float* w_enc, float* d_b_pre,
                        unsigned int* ticket, long long dead_threshold, long long* dead_count,
                        const long long* seq, long long* mailbox, wsae_stream_t stream);

/* ---- K2: k-sparse decode + MSE + L0 + fired stamps (sae/model.py:116,129,145,148,174-181) -----
 * recon = sum_j relu(val_j) * W_decT[idx_j,:] + b_dec (+ b_pre);  resid = recon - target.
 * stats (16 bytes, caller-zeroed): { double sse; uint64 l0_count }.
 * If last_activated/step_count are non-NULL (training mode), last_activated[f] = *step_count + 1
 * for every feature with a selected value > 0 (the +1 on step_count itself is
 * wsae_counters_update).  w_decT is [F,d] fp32 (w_is_bf16 = 0) or bf16 (1). */
int wsae_decode_mse(const float* target, const void* w_decT, int w_is_bf16, const float* b_dec,
                    const float* b_pre /*nullable*/, const int32_t* idx, const float* val, int B,
                    int d, int F, int k, float* resid /*nullable [B,d]*/,
                    float* recon /*nullable [B,d]*/, void* stats /*nullable*/,
                    long long* last_activated /*nullable [F]*/,
                    const long long* step_count /*nullable*/, wsae_stream_t stream);

/* ---- K3: sparse backward (autograd of sae/model.py:108-145, run at sae/training.py:184) -------
 * s = coef * (*grad_out) with coef = 2 / (B_total * d).  Accumulates (+=) into the caller-zeroed
 * gradient buffers; any of d_w_enc / d_w_decT / d_b_enc / d_b_dec / dpre_val may be NULL to skip
 * that output.  dpre_val[b,j] = [val>0] * s * (resid_b . W_decT[idx,:]).  d % 4 == 0.
 * resid_bf16 (optional) receives bf16(resid), the dense operand of the K4 dW_decT GEMM. */
int wsae_backward_sparse(const float* resid, const float* x /*nullable if !d_w_enc*/,
                         const float* b_pre /*nullable*/, const void* w_decT, int w_is_bf16,
                         const int32_t* idx, const float* val, const float* grad_out /*nullable*/,
                         float coef, int B, int d, int F, int k, float* d_w_enc /*[F,d]*/,
                         float* d_w_decT /*[F,d]*/, float* d_b_enc /*[F]*/, float* d_b_dec /*[d]*/,
                         float* dpre_val /*[B,k]*/, void* resid_bf16 /*nullable bf16 [B,d]*/,
                         wsae_stream_t stream);
/* ---- K23: K2 and the sparse part of K3 fused into one pass over the gathered decoder rows -------
 * (sae/model.py:115-116,129,145,148,174-181 + the dv / bias part of its autograd).  For the train
 * step where grad_out is known when the forward runs (loss.backward() with grad_output = 1, i.e.
 * the CUDA-graphed SAETrainer.train_step).  One warp per activation row; the k selected decoder
 * rows (bf16 shadow) are loaded into registers once, 128 columns at a time, and used for both the
 * reconstruction and the k dot products (bf16 x bf16 -> fp32 FHFMA against the bf16-rounded
 * residual, the same rounding K4 consumes).  Outputs as in wsae_decode_mse / wsae_backward_sparse
 * (weight gradients are left to K4); resid / resid_bf16 / stats / last_activated / d_b_enc /
 * d_b_dec / dpre_val may each be NULL.  d_b_enc and d_b_dec are accumulated (+=).
 * k ranges: k <= 32 one warp per row; 32 < k <= 256 (d % 128 == 0 only) a team of ceil(k / 32)
 * warps per row, each holding 32 of the k gathered rows, meeting once per 64 columns to form the
 * residual.  Returns WSAE_E_UNSUPPORTED for an fp32 decoder, d % 8 != 0, k > 256, or k > 32 with
 * d % 128 != 0: use K2 + K3 then.  The deterministic form (wsae_decode_backward_det, or a non-NULL
 * det_ws) covers the same shapes. */
int wsae_decode_backward(const float* target, const void* w_decT, int w_is_bf16,
                         const float* b_dec, const float* b_pre /*nullable*/, const int32_t* idx,
                         const float* val, const float* grad_out /*nullable*/, float coef, int B,
                         int d, int F, int k, float* resid, void* resid_bf16, void* stats,
                         long long* last_activated, const long long* step_count, float* d_b_enc,
                         float* d_b_dec, float* dpre_val, wsae_stream_t stream);
/* As wsae_decode_backward, with the target matrix named by a device-resident pointer slot
 * (*target_at: 16-byte aligned, B x d fp32, read when the kernel runs; see
 * wsae_pack_activations_at). */
int wsae_decode_backward_at(const float* const* target_at, const void* w_decT, int w_is_bf16,
                            const float* b_dec, const float* b_pre /*nullable*/,
                            const int32_t* idx, const float* val, const float* grad_out /*nullable*/,
                            float coef, int B, int d, int F, int k, float* resid, void* resid_bf16,
                            void* stats, long long* last_activated, const long long* step_count,
                            float* d_b_enc, float* d_b_dec, float* dpre_val, wsae_stream_t stream);
/* As wsae_decode_backward_at, target row of batch row r = (*target_at)[(*rows_at)[r], :]
 * (see wsae_pack_activations_rows_at). */
int wsae_decode_backward_rows_at(const float* const* target_at, const long long* const* rows_at,
                                 const void* w_decT, int w_is_bf16, const float* b_dec,
                                 const float* b_pre /*nullable*/, const int32_t* idx, const float* val,
                                 const float* grad_out /*nullable*/, float coef, int B, int d, int F,
                                 int k, float* resid, void* resid_bf16, void* stats,
                                 long long* last_activated, const long long* step_count,
                                 float* d_b_enc, float* d_b_dec, float* dpre_val, wsae_stream_t stream);
/* Slot form for any target dtype: *target_at holds elements of type x_dtype (16-byte aligned); rows_at
 * nullable (as in wsae_decode_backward_rows_at); det_ws nullable (non-NULL: wsae_decode_backward_det's
 * deterministic accumulation, finished by wsae_det_finish).  Covers every K23 form (warp, staged, tensor,
 * team). */
int wsae_decode_backward_typed(const void* const* target_at, const long long* const* rows_at /*nullable*/,
                               int x_dtype, const void* w_decT, int w_is_bf16, const float* b_dec,
                               const float* b_pre /*nullable*/, const int32_t* idx, const float* val,
                               const float* grad_out /*nullable*/, float coef, int B, int d, int F, int k,
                               float* resid, void* resid_bf16, void* stats, long long* last_activated,
                               const long long* step_count, float* d_b_enc, float* d_b_dec, float* dpre_val,
                               long long* det_ws /*nullable*/, wsae_stream_t stream);
/* out[idx[b,j], :] += vals[b,j] * (rows[b,:] - center): the encoder weight gradient as a sparse
 * scatter when the input width differs from the decoder width (transcoders); dr % 4 == 0. */
int wsae_scatter_rows(const float* rows, const float* center /*nullable*/, const int32_t* idx,
                      const float* vals, int B, int dr, int F, int k, float* out /*[F,dr]*/,
                      wsae_stream_t stream);
/* db_pre = db_dec - db_enc . W_enc  (overwrites d_b_pre). */
int wsae_bpre_grad(const float* d_b_dec, const float* d_b_enc, const float* w_enc, int F, int d,
                   float* d_b_pre, wsae_stream_t stream);
/* dx = dpre . W_enc (- g if subtract_g): only needed when the input requires grad. */
int wsae_input_grad(const float* resid, const float* w_enc, const int32_t* idx,
                    const float* dpre_val, const float* grad_out, float coef, int B, int d, int F,
                    int k, int subtract_g, float* dx, wsae_stream_t stream);

/* ---- K4: tensor-core weight gradients (autograd `mm`s of sae/model.py:111,129 at training.py:184)
 * OUT[F,d] += alpha * (*grad_out) * S^T . R, with S the k-sparse [B,F] matrix given as (idx, value)
 * entries and R a dense bf16 [B,d] matrix (row pitch r_pitch_elems, a multiple of 8, base 16-byte
 * aligned); tcgen05 GEMM (M = 128 features, N = d, K = batch rows) whose sparse operand is expanded
 * to dense bf16 tiles in shared memory only.  Used for
 *   dW_enc  : values = dpre_val,  R = bf16(x - b_pre)   (the packed activations of K0, terms = 1)
 *   dW_decT : values = relu(val), R = bf16(resid), alpha = 2 / (B_total * d)
 * wsae_bucket_by_tile groups the active entries (val > 0) by (64-row chunk, 128-feature tile); the
 * entries of chunk c live in its own segment [c * 64 * k, ...) of the entry arrays:
 *   offsets  int32 [n_chunks * (n_ft + 1)]  (cell (c, ft) owns [offsets[c*(n_ft+1)+ft], offsets[c*(n_ft+1)+ft+1]))
 *   ent_meta uint32 [B*k]  = row_in_chunk | feature_in_tile << 8
 *   ent_a / ent_b float [B*k] = dpre_val / val of the entry
 * with n_chunks, n_ft from wsae_bucket_cells.  OUT is accumulated with red.global.add (split-K). */
int wsae_bucket_cells(int B, int F, int* n_chunks, int* n_ft);
int wsae_bucket_by_tile(const int32_t* idx, const float* val, const float* dpre, int B, int F,
                        int k, int* offsets, uint32_t* ent_meta, float* ent_a, float* ent_b,
                        wsae_stream_t stream);
int wsae_wgrad_gemm(const void* r_bf16, int r_pitch_elems, int B, int F, int d, const int* offsets,
                    const uint32_t* ent_meta, const float* ent_val, const float* grad_out /*nullable*/,
                    float alpha, float* out /*[F,d]*/, wsae_stream_t stream);

/* ---- K5: elementwise / reductions ------------------------------------------------------------
 * renorm: rows of W_decT /= max(||row||, eps)  (sae/model.py:91-96, F.normalize(dim=0), eps 1e-12);
 *         optionally refreshes the bf16 shadow in the same pass.
 * counters: if bump, *step_count += 1 (model.py:174); *dead_count = #{f: step - last[f] > thr}
 *         (model.py:183-195). */
int wsae_renorm_decoder(float* w_decT, int F, int d, float eps, void* bf16_shadow /*nullable*/,
                        wsae_stream_t stream);
int wsae_counters_update(const long long* last_activated, long long* step_count, int F,
                         long long threshold, int bump, long long* dead_count /*nullable*/,
                         wsae_stream_t stream);
/* wsae_counters_update, then the step's metrics posted to a host mailbox: mailbox[0..2] = {stats2[0]
 * (SSE, f64 bits), stats2[1] (L0 count), dead count}, a system-scope fence, mailbox[3] = *seq.
 * `mailbox` is 4 x int64 of page-locked host memory (device-accessible at the same address under
 * UVA); `seq` a device int64 the caller bumps per step.  The host polls mailbox[3] instead of
 * synchronising with the stream: the five `.item()` syncs of sae/training.py:206-214 become one
 * poll that returns while the rest of the step is still running. */
int wsae_counters_update_post(const long long* last_activated, long long* step_count, int F,
                              long long threshold, int bump, long long* dead_count /*nullable*/,
                              const long long* stats2 /*nullable*/, const long long* seq,
                              long long* mailbox, wsae_stream_t stream);
/* hidden[B,F] = scatter(relu(val)) (sae/model.py:115-116) for API callers that need it dense. */
int wsae_densify_hidden(const int32_t* idx, const float* val, int B, int F, int k, float* hidden,
                        wsae_stream_t stream);
int wsae_cast_bf16(const float* src, void* dst_bf16, long long n, wsae_stream_t stream);
/* *out += sum(g^2) (double): building block of clip_grad_norm_ (sae/training.py:188-191). */
int wsae_sumsq(const float* g, long long n, double* out, wsae_stream_t stream);
/* Clip scale + AdamW in one pass (sae/training.py:187-194, torch.optim.AdamW semantics).
 * hyper (device, 8 floats) = {lr, beta1, beta2, eps, weight_decay, 1-beta1^t, sqrt(1-beta2^t),
 * max_norm}; grad_sumsq (device double, nullable) = total squared grad norm over all params. */
int wsae_fused_adamw(float* p, const float* grad, float* m, float* v, long long n,
                     const float* hyper, const double* grad_sumsq, wsae_stream_t stream);

/* The same update for up to 8 parameter tensors in ONE launch.  row_len > 0 marks a
 * [n / row_len, row_len] matrix whose rows are re-normalised to unit L2 norm (clamped at
 * renorm_eps) right after the update: optimizer.step() followed by normalize_decoder_weights()
 * (sae/training.py:193-198, sae/model.py:91-96) in a single pass over the decoder.  `tensors` is a
 * HOST array (copied into the kernel arguments); the pointers inside are device pointers.
 * flags bit 0 (WSAE_ADAMW_PROJECT_GRAD, rows only; NOT in the reference, default off): before the
 * update the row's gradient loses its component along the decoder row, g -= (g.w / w.w) w
 * (BASELINE north_star "gradient projection"); parity tests run with it off. */
#define WSAE_ADAMW_PROJECT_GRAD 1
typedef struct {
  float* p;
  const float* g;
  float* m;
  float* v;
  long long n;
  int row_len;
  int flags;
} wsae_adamw_tensor_t;
int wsae_adamw_multi(const wsae_adamw_tensor_t* tensors, int count, const float* hyper,
                     const double* grad_sumsq, float renorm_eps, wsae_stream_t stream);

/* ---- Per-feature top-K activating examples (analysis/feature_viz.py:94-158 TopKTracker.update,
 *      :425-484 collect_top_activations) --------------------------------------------------------
 * Consumes the sparse code the hot path produces.  Entries i = 0..n-1 are (feat[i], val[i]) with
 * row(i) = rows ? rows[i] : i / k (k = entries per row of an [B, k] TopK result); an entry counts
 * when val > 0 (and 0 <= feat < F).  Per feature the K largest values seen so far are kept with
 * their sample id (sample_ids ? sample_ids[row] : sample_base + row) and position
 * (pos_ids ? pos_ids[row] : 0): top_val [F,K] descending with -inf = empty, top_sample int64 [F,K],
 * top_pos int32 [F,K] (-1 = empty), top_count int32 [F].  An entry displaces the current K-th only
 * if STRICTLY larger (the reference's heap rule), so among equal values the earlier arrival -
 * earlier call, then lower row - stays.  *total += number of counted entries
 * (TopKTracker.total_activations).  K <= 32, n < 2^31.  ws: wsae_feature_topk_workspace bytes. */
int wsae_feature_topk_workspace(long long n, int F, unsigned long long* bytes);
int wsae_feature_topk_update(const int32_t* feat, const float* val, const int32_t* rows /*nullable*/,
                             long long n, int k, const long long* sample_ids /*nullable*/,
                             long long sample_base, const int32_t* pos_ids /*nullable*/, int F, int K,
                             float* top_val, long long* top_sample, int32_t* top_pos,
                             int32_t* top_count, unsigned long long* total, void* ws,
                             unsigned long long ws_bytes, wsae_stream_t stream);

/* ---- Activation extraction: final LayerNorm of hooked Whisper hidden states, flattened
 *      (sae/hooks.py:85-86,103-104 `layer_norm(hidden_states)`, :213-230 flatten_activations) ----
 * out[r, :] = (x[r, :] - mean_r) * rsqrt(var_r + eps) * gamma + beta  for r in [0, rows): biased
 * variance, fp32 arithmetic (torch.nn.LayerNorm); x is [rows, d] with row pitch in_pitch_elems,
 * in_dtype 0 = float32 / 1 = bfloat16 / 2 = float16; out is float32 with row pitch
 * out_pitch_elems - pass `matrix + row0 * pitch` to append a batch to a [N, d] activation matrix
 * (flatten + concatenate of hooks.py / feature_cache.py:283-300).  gamma / beta nullable.  d <= 4096. */
int wsae_layernorm_rows(const void* x, int in_dtype, long long rows, int d, long long in_pitch_elems,
                        const float* gamma /*nullable*/, const float* beta /*nullable*/, float eps,
                        float* out, long long out_pitch_elems, wsae_stream_t stream);
/* As wsae_layernorm_rows, writing elements of type out_dtype: the statistics and the normalised value are
 * fp32 as above, rounded to nearest at the store. */
int wsae_layernorm_rows_typed(const void* x, int in_dtype, long long rows, int d, long long in_pitch_elems,
                              const float* gamma /*nullable*/, const float* beta /*nullable*/, float eps,
                              void* out, int out_dtype, long long out_pitch_elems, wsae_stream_t stream);

/* ---- Splicing a TopK SAE into Whisper's forward pass (sae/splice.py) ---------------------------
 * A site's layer output row h [d] (dtype h_dtype), its mean mu and biased variance var, r = rsqrt(var + eps):
 *   x      = (h - mu) * r * gamma + beta                 (the fp32 formula of wsae_layernorm_rows)
 *   (i, v) = TopK_k(pack(x - b_pre) . W'^T)             (wsae_encode_topk*, terms = 1)
 *   a_j    = relu(v_j), rounded to bf16                  (K2's convention)
 *   recon  = sum_j a_j W_dec[i_j] + b_dec + b_pre        (bf16 decoder shadow, fp32 accumulation)
 *   recon' = sum_j gain[i_j] a_j W_dec[i_j] + b_dec + b_pre + steer
 *   mode 0 (replace): h' = mu + ((recon' - beta) / gamma) / r
 *   mode 1 (error)  : h' = h + ((recon' - recon) / gamma) / r; an element whose difference is exactly 0 is
 *                     written back with h's bits.  recon' - recon is accumulated directly, as
 *                     steer + sum (gain - 1) a_j W_dec[i_j] over the entries whose gain is not 1.
 * h' is written in h's dtype, rounded to nearest.  Without the LayerNorm (row_stats == NULL in the decode;
 * pack with wsae_pack_activations_typed) x = h and the inverse map is the identity.
 *
 * wsae_splice_pack: a_packed = pack_activations(LN(h), b_pre, terms = 1) bit for bit ([Bp, Kp] bf16, rows
 *   >= N zero, Bp % 128 == 0) and row_stats [N, 2] = (mu, r) float32; h is [N, d] with row pitch d.
 * wsae_splice_decode: out [N, d] (h's dtype; may not alias h).  idx / val [N, k] from K1, any k, padding
 *   (-inf, -1) allowed.  gain [F] / steer [d] / gamma / beta nullable (1 / 0).  Accumulators, nullable,
 *   caller-zeroed, added to: stats {double sse (unmodified recon against x); double sum x^2; uint64 l0},
 *   x_sum double [d], feature_count int64 [F] (rows in which each feature fired).
 * Both: d % 8 == 0, d <= 4096 (WSAE_E_UNSUPPORTED above), pointers 16-byte aligned. */
int wsae_splice_pack(const void* h, int h_dtype, int N, int Bp, int d, const float* gamma /*nullable*/,
                     const float* beta /*nullable*/, float eps, const float* b_pre /*nullable*/,
                     void* a_packed /*bf16 [Bp,Kp]*/, float* row_stats /*[N,2]*/, wsae_stream_t stream);
int wsae_splice_decode(const void* h, int h_dtype, const float* row_stats /*nullable*/,
                       const float* gamma /*nullable*/, const float* beta /*nullable*/,
                       const void* w_decT_bf16 /*[F,d]*/, const float* b_dec, const float* b_pre /*nullable*/,
                       const int32_t* idx, const float* val, const float* gain /*nullable*/,
                       const float* steer /*nullable*/, int N, int d, int F, int k, int mode, void* out,
                       void* stats /*nullable*/, double* x_sum /*nullable*/,
                       long long* feature_count /*nullable*/, wsae_stream_t stream);

/* ---- deterministic accumulation mode (SAETrainer(..., deterministic=True)) ----------------------
 * The default kernels add their cross-row / split-K partial sums with float atomics in arrival
 * order, so two runs of the same step differ in the last bits.  These forms are bit-reproducible:
 *   wsae_decode_backward_det : K23 with db_enc / db_dec / SSE accumulated as fixed-point int64 in
 *       det_ws [F + d + 1] (caller-zeroed; addends are the unscaled dot products, |.| < 2^10);
 *       wsae_det_finish converts: d_b_enc += s*sum, d_b_dec += s*sum, stats.sse += sum,
 *       s = coef * (*grad_out).  target (direct) or target_at (slot) names the matrix; rows_at nullable.
 *       Shapes: k <= 32 with d % 8 == 0, and 32 < k <= 256 with d % 128 == 0 (the team form: db_dec
 *       and SSE are summed per block in team / warp order before the fixed-point add).  A feature
 *       gets at most one db_enc addend per row at any k, so the int64 headroom does not depend on k.
 *   wsae_wgrad_gemm_det      : K4 with one partial slab per k split in ws (wsae_wgrad_gemm_workspace
 *       bytes; 0 = no split) and an ordered reduction instead of red.global.add.
 *   wsae_sumsq_det           : per-block partials in ws (wsae_sumsq_det_blocks() doubles), ordered sum.
 *   wsae_bpre_grad_det       : per-256-feature partial rows in ws (ceil(F/256)*d floats), ordered sum. */
int wsae_decode_backward_det(const float* target /*nullable*/, const float* const* target_at /*nullable*/,
                             const long long* const* rows_at /*nullable*/, const void* w_decT,
                             int w_is_bf16, const float* b_dec, const float* b_pre /*nullable*/,
                             const int32_t* idx, const float* val, const float* grad_out /*nullable*/,
                             float coef, int B, int d, int F, int k, float* resid, void* resid_bf16,
                             void* stats, long long* last_activated, const long long* step_count,
                             float* d_b_enc, float* d_b_dec, float* dpre_val, long long* det_ws,
                             wsae_stream_t stream);
int wsae_det_finish(const long long* det_ws, int F, int d, const float* grad_out /*nullable*/, float coef,
                    float* d_b_enc /*nullable*/, float* d_b_dec /*nullable*/, void* stats /*nullable*/,
                    wsae_stream_t stream);
int wsae_wgrad_gemm_workspace(int B, int F, int d, unsigned long long* bytes);
int wsae_wgrad_gemm_det(const void* r_bf16, int r_pitch_elems, int B, int F, int d, const int* offsets,
                        const uint32_t* ent_meta, const float* ent_val, const float* grad_out /*nullable*/,
                        float alpha, float* out /*[F,d]*/, float* ws, unsigned long long ws_bytes,
                        wsae_stream_t stream);
int wsae_sumsq_det_blocks(void);
int wsae_sumsq_det(const float* g, long long n, double* ws, double* out, wsae_stream_t stream);
int wsae_bpre_grad_det(const float* d_b_dec, const float* d_b_enc, const float* w_enc, int F, int d,
                       float* d_b_pre, float* ws, wsae_stream_t stream);

/* ---- experiments only (tools/bench_k1.py); not part of the product path -----------------------
 * variant: 0 = per-batch choice (default: CTA pairs from 1024 rows), 1 = one epilogue warp per TMEM lane
 * quarter, 2 = scanner + selector warps (single CTA), 3 = scanner + selector on CTA pairs (cta_group::2);
 * mode (variant 1): 0 = product, 1 = release the accumulators unread (GEMM pipeline alone),
 * 2 = scan without compaction; counters: device buffer u64 [grid][8][8] for the scanner/selector
 * wait breakdown (NULL = off). */
int wsae_debug_encode_variant(int variant);
int wsae_debug_encode_mode(int mode);
int wsae_debug_encode_counters(void* device_buf);
int wsae_debug_wgrad_cluster(int max_cluster_size); /* 1, 2 (default), 4, 8: upper bound for wsae_wgrad_gemm's cluster */
int wsae_debug_decode_backward_general(int mode);   /* wsae_decode_backward kernel choice: 0 = per-shape (default), 1 = general, 2 = mma.sync dots, 3 = cp.async staged (A/B runs) */

#ifdef __cplusplus
}
#endif
#endif /* WSAE_H_ */
