/* rnvp.h -- C ABI of the B200-native RealNVP hot path (librnvp_b200.so).
 *
 * Drop-in boundary for hse-cs/probaforms' RealNVP path.  The reference has no
 * native code: its hot path is Python calling torch eager ops.  Each entry
 * point below replaces the reference interface cited next to it (paths are
 * relative to the reference repo root); INTEGRATION.md shows the ctypes stub a
 * maintainer would add on the reference side.
 *
 * Conventions
 *  - plain C types only; every pointer named d_* is a DEVICE pointer to
 *    contiguous fp32 (or int64 where stated) memory owned by the caller (torch);
 *    the library never allocates or frees caller-visible memory.  The opaque
 *    descriptor owns a few KB of device tables (its per-tile op programs).
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it.  The per-tile programs of the
 *    FP32 kernels for the whole flow are built and uploaded by rnvp_desc_create (synchronous, once), so
 *    rnvp_forward / rnvp_inverse / rnvp_sample / rnvp_backward / rnvp_adam_step over the full layer range
 *    neither allocate nor synchronise and are CUDA-graph capturable; a call on a layer SUB-range
 *    (RealNVPLayer.f / .g) builds its program on first use (one cudaMalloc + synchronous copy, then cached).
 *  - the only process-global mutable state is the development trace pointer of rnvp_debug_set_trace;
 *    everything else lives in the descriptor (guarded by a mutex) or on the caller's stream.
 *  - every function returns 0 on success, a negative RNVP_E* code for argument /
 *    planning errors, or a positive cudaError_t.  rnvp_last_error() returns a
 *    thread-local message.  Nothing throws, exits, or falls back to the CPU.
 *  - parameters cross the boundary in the reference's own layout: one flat fp32
 *    buffer in `nf.parameters()` order, per coupling layer i
 *    nn_t.0.weight [h0, D+Cd], nn_t.0.bias [h0], ..., nn_t.{2n}.weight [D, h_last],
 *    nn_t.{2n}.bias [D], then the same for nn_s  (probaforms/models/realnvp.py:69-70,
 *    gen_network realnvp.py:19-43).  rnvp_pack_params() converts it to the
 *    kernel-private mask-compacted "packed" layout; gradients come back through
 *    rnvp_unpack_grads() with exact zeros on masked rows/columns, as autograd
 *    produces them in the reference.
 */
#ifndef RNVP_H
#define RNVP_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rnvp_desc rnvp_desc;

enum {
  RNVP_OK = 0,
  RNVP_EINVAL = -1,      /* bad argument */
  RNVP_ESHAPE = -2,      /* flow shape cannot be planned (e.g. shared-memory budget) */
  RNVP_ENODEVICE = -3,   /* no sm_100 device / wrong architecture */
  RNVP_EALLOC = -4
};
enum { RNVP_ACT_TANH = 1, RNVP_ACT_RELU = 2 };   /* realnvp.py:32-37 */

/* Build the descriptor of a flow on the CURRENT CUDA device.
 * Replaces RealNVP._model_init's layer construction (realnvp.py:195-204):
 * L coupling layers over var_size=D, cond_size=Cd (0 when C is None), conditioner
 * hidden widths hidden[0..n_hidden-1], mask_i[j] = (j+i)%2 (realnvp.py:199). */
int rnvp_desc_create(int D, int Cd, int L, int n_hidden, const int* hidden, int act, rnvp_desc** out);
void rnvp_desc_destroy(rnvp_desc* d);

/* sizes, in floats */
int64_t rnvp_param_count(const rnvp_desc* d);    /* P: flat reference-layout parameters */
int64_t rnvp_packed_count(const rnvp_desc* d);   /* kernel-private packed layouts (all kernel families) */
int64_t rnvp_grad_count(const rnvp_desc* d);     /* floats of the packed gradient accumulator d_gpacked */
/* bytes of scratch rnvp_backward needs for a batch of N rows: the per-CTA x_T stash of the fused FP32 kernel
 * (independent of N, stays L2 resident); on the tensor-core fit paths the per-layer (x_T, s) stash plus the
 * activation records, Npad*L*(D + rnvp_wgrad_record_floats)*4 bytes (Npad = N rounded up to whole row tiles) */
int64_t rnvp_workspace_bytes(const rnvp_desc* d, int64_t N);
/* offsets[2*k], offsets[2*k+1] = (float offset, numel) of the k-th tensor of nf.parameters();
 * n = 4*(n_hidden+1)*L entries pairs.  Returns the number of tensors. */
int rnvp_param_tensors(const rnvp_desc* d, int64_t* offsets, int max_tensors);
/* plan introspection: mode 0 forward, 1 inverse, 2 fused forward+backward, 4 = "is the whole fit step on the tensor
 * cores" (kernel_family 2 iff yes; mode 3 is not used and gives RNVP_EINVAL); rows per CTA tile, shared memory, ops per
 * tile of the FP32 program, kernel family (0 tile, 1 small-flow, 2 tcgen05) */
int rnvp_plan_info(const rnvp_desc* d, int mode, int* tile_rows, int* smem_bytes, int* n_ops, int* kernel_family);

/* flat (reference layout) -> packed; run after every parameter update */
int rnvp_pack_params(const rnvp_desc* d, const float* d_flat, float* d_packed, void* stream);
/* packed gradient accumulator -> flat reference layout (masked entries written as exact 0) */
int rnvp_unpack_grads(const rnvp_desc* d, const float* d_gpacked, float* d_gflat, void* stream);

/* Forward pass = body of NormalizingFlow.log_prob before the mean (nflow.py:107-115) over
 * layers [layer_begin, layer_end): z, per-row sum of log|det J|, and
 * logp = logdet + MultivariateNormal(0,I).log_prob(z).  Any of d_z/d_logdet/d_logp may be NULL.
 * layer_end - layer_begin == 1 is RealNVPLayer.f (realnvp.py:73-101).  d_C NULL iff Cd == 0.
 * d_idx (int64[N], may be NULL) gathers rows: row r reads X[idx[r]], C[idx[r]]. */
int rnvp_forward(const rnvp_desc* d, const float* d_packed, const float* d_X, const float* d_C,
                 const int64_t* d_idx, int64_t N, int layer_begin, int layer_end,
                 float* d_z, float* d_logdet, float* d_logp, void* stream);

/* Inverse pass = NormalizingFlow.sample after the prior draw (nflow.py:142-143): layers
 * [layer_begin, layer_end) applied in REVERSE order to the latent rows d_Y (the prior sample);
 * one layer is RealNVPLayer.g (realnvp.py:104-129). */
int rnvp_inverse(const rnvp_desc* d, const float* d_packed, const float* d_Y, const float* d_C,
                 int64_t N, int layer_begin, int layer_end, float* d_X, void* stream);

/* NormalizingFlow.sample in one launch (nflow.py:141-143): the prior draw X = prior.sample((n,)) is generated inside the
 * inverse kernel instead of being written to and read back from device memory.  Latent element (row, j) is a pure
 * function of (seed, row_offset + row, j) -- Philox4x32-10 + Box-Muller, csrc/rnvp_philox.cuh -- so a row block gives
 * the same rows whichever GPU or launch produces it: shard a request of n rows over GPUs by passing each shard its
 * first global row as row_offset (no communication).  rnvp_inverse stays the parity mode (caller-supplied noise). */
int rnvp_sample(const rnvp_desc* d, const float* d_packed, const float* d_C, int64_t N, uint64_t seed,
                int64_t row_offset, float* d_X, void* stream);

/* Fused forward + backward of  out = scale * sum_rows logp(row)  (loss.backward() of
 * loss = -nf.log_prob(X, C), realnvp.py:246-250, is scale = -1/N).  Weight gradients are ACCUMULATED into
 * d_gpacked (caller zeroes it), sum_rows logp is accumulated into d_logp_sum (1 float, may be NULL), per-row
 * logp optionally written.  Kernel families: small flows and the generic FP32 tile kernel recompute the
 * hidden activations in the backward sweep (nothing but x_T per layer is kept); the tensor-core fit path
 * (tcgen05-eligible flows with D <= 64, or with H a multiple of 128) hands h, u and delta2 of every
 * (layer, row) to the weight-gradient sweep through activation records in d_workspace (see
 * rnvp_wgrad_sweep), which is why rnvp_workspace_bytes grows with N there. */
int rnvp_backward(const rnvp_desc* d, const float* d_packed, const float* d_X, const float* d_C,
                  const int64_t* d_idx, int64_t N, float scale, float* d_gpacked, float* d_logp_sum,
                  float* d_logp, void* d_workspace, int64_t workspace_bytes, void* stream);

/* torch.optim.Adam step (realnvp.py:205-207, 251; betas/eps as constructed there) on the flat
 * parameters, refreshing d_packed in the same pass.  The gradient is read from the packed
 * accumulator d_gpacked, or, when d_gflat_in is non-NULL, from a reference-layout gradient (the
 * .grad tensors autograd filled); grad_scale multiplies it first (e.g. 1/world_size after an
 * all-reduce).  step is the 1-based step count; scalar hyper-parameters are doubles because torch
 * does the bias-correction arithmetic in Python doubles.  d_gflat_out (may be NULL) receives the
 * reference-layout gradient.  zero_gpacked != 0 re-zeroes the accumulator entries it consumed
 * (opt.zero_grad(), realnvp.py:249).  If d_loss_src is non-NULL, *d_loss_dst = *d_loss_src *
 * loss_scale (loss_history entry, realnvp.py:254) and *d_loss_src is re-zeroed with the gradients. */
int rnvp_adam_step(const rnvp_desc* d, float* d_flat, float* d_packed, float* d_gpacked,
                   const float* d_gflat_in, float* d_exp_avg, float* d_exp_avg_sq, float* d_gflat_out,
                   float grad_scale, double lr, double beta1, double beta2, double eps,
                   double weight_decay, int64_t step, int zero_gpacked, float* d_loss_src,
                   float* d_loss_dst, float loss_scale, void* stream);

/* One epoch of the reference's fit loop (realnvp.py:238-254) as ONE call: for every consecutive slice of `batch_size`
 * entries of the epoch's row order d_perm[n] (the last partial batch is kept): rnvp_backward with scale = -1/nb, then
 * rnvp_adam_step (step count step0 + 1, step0 + 2, ...), the step's loss written to d_losses[s].  Same arithmetic as the
 * two calls it wraps, bit for bit; it removes the host-side per-step overhead, which dominates README-sized batches, and
 * for small flows whose batch fits one 32-row tile (the reference's default batch_size) each step is ONE launch: the
 * fit kernel applies the Adam update, refreshes d_packed and hands the loss off itself (the step's gradient is already in
 * its shared memory; 16 us per step on B200 against 23 us for the two launches).  Single GPU (no all-reduce between the
 * two).  d_gpacked and *d_loss_slot must be zero on entry and are zero again on return. */
int rnvp_fit_epoch(const rnvp_desc* d, float* d_flat, float* d_packed, float* d_gpacked, float* d_exp_avg, float* d_exp_avg_sq,
                   const float* d_X, const float* d_C, const int64_t* d_perm, int64_t n, int64_t batch_size, double lr,
                   double beta1, double beta2, double eps, double weight_decay, int64_t step0, float* d_loss_slot,
                   float* d_losses, void* d_workspace, int64_t workspace_bytes, void* stream);

/* Weight-gradient sweep from stored activations (last part of a fit step on the tcgen05 path): for every layer
 * dW1 += delta1^T u, db1 += sum delta1, dW2 += delta2^T h, db2 += sum delta2 (sums over rows), accumulated into
 * d_gpacked, with delta1 = (delta2 W2) * act'(h) recomputed from d_packed.  One record of
 * rec = rnvp_wgrad_record_floats(d) floats per (layer, row):
 * h [2][H] (nn_t | nn_s) | u = [x_K, c, 0..] (ceil8(D/2+Cd)) | delta2 [2][D/2],
 * stored in blocks of 32 rows as d_records[L][Npad/32][rec/4][32][4]: float4 column group q of row r of a block sits
 * in slot (r ^ (q & 7)).  Npad is a multiple of 32; padding rows must hold zeros in delta1 / delta2.
 * Flows whose fit step runs on the tensor cores: tcgen05-eligible flows (see rnvp_set_path) with D <= 64, or with H a
 * multiple of 128 (one 128-lane block of hidden units per CTA, rnvp_wgrad_tc.cu). */
int rnvp_wgrad_record_floats(const rnvp_desc* d);
int rnvp_wgrad_sweep(const rnvp_desc* d, const float* d_packed, int64_t Npad, const float* d_records, float* d_gpacked,
                     void* stream);

/* Kernel-family selection for rnvp_forward / rnvp_inverse: 0 = auto (tcgen05 TF32x3 kernels where the shape is
 * eligible -- one hidden layer, 8 < D <= 128, Cd <= 16 (D <= 64) or 32, H a multiple of 32, and for D <= 32 the
 * whole-layer weight images within the shared memory of one CTA --, else the small-flow or FP32 tile kernels),
 * 1 = FP32-FMA kernels only, 2 = same as auto.  rnvp_plan_info reports the family chosen (0 tile, 1 small-flow,
 * 2 tcgen05). */
int rnvp_set_path(rnvp_desc* d, int path);

/* Host-side row order of one epoch, produced incrementally (replaces the per-epoch DataLoader(shuffle=True) of
 * realnvp.py:237: RandomSampler -> torch.randperm(n, generator=Generator().manual_seed(seed)); bit-identical to it).
 * `out` is a caller-owned HOST buffer of n int64 (pinned memory recommended).  rnvp_perm_advance finalises
 * out[0 .. upto) and returns the number of final entries, so the first batches can be consumed while a helper thread is
 * still shuffling the tail.  n must be below 2^32/20 (torch uses another scheme beyond: RNVP_ESHAPE).  No device work. */
typedef struct rnvp_perm rnvp_perm;
int rnvp_perm_create(uint64_t seed, int64_t n, int64_t* out, rnvp_perm** p);
int64_t rnvp_perm_advance(rnvp_perm* p, int64_t upto);
void rnvp_perm_destroy(rnvp_perm* p);

/* Host-side ingestion / egress helpers (no device work; HOST pointers).  rnvp_host_gather_xc writes
 * dst_x[r][0..width_x) = (float) src_x[idx ? idx[r] : row0 + r][0..width_x) for r in [0, n), and the same rows of src_c
 * into dst_c in the same pass over idx; src_c may be NULL (X rows only: c_is_f64, width_c and dst_c are then ignored).
 * These are the rows of one optimisation step or one upload chunk, converted from the caller's float64 (x_is_f64 /
 * c_is_f64 != 0) or float32 arrays -- torch.tensor(X, dtype=float32) of realnvp.py:226-228 fused with the batch gather
 * of realnvp.py:237 -- into (pinned) staging buffers, on up to `threads` host threads.  A staging buffer is written with
 * non-temporal stores when it is 16-byte aligned and its width % 4 == 0: its next reader is the GPU's DMA engine, and an
 * upload whose source lines are dirty in many cores' caches runs at a quarter of the bus rate.  rnvp_host_copy is a
 * multi-threaded memcpy (the .cpu().numpy() of realnvp.py:281 into a fresh pageable array; RealNVP.sample uses it only
 * beyond the pinned result pool's cap). */
int rnvp_host_gather_xc(const void* src_x, int x_is_f64, int64_t width_x, const void* src_c, int c_is_f64, int64_t width_c,
                           const int64_t* idx, int64_t row0, int64_t n, float* dst_x, float* dst_c, int threads);
int rnvp_host_copy(void* dst, const void* src, int64_t bytes, int threads);

/* Development aid: when d_buf (device, >= 43 int64) is non-null and the library was built with -DRNVP_WG_TRACE, every
 * role of CTA 0 of the tcgen05 weight-gradient sweep writes the cycles it spent in each of its mbarrier waits
 * (d_buf[role * 8 + wait site]; d_buf[40..42]: CTA 0's rows, rows per stage, cycles from entry to the end of its flush;
 * see rnvp_wgrad_tc.cu; tools/trace_wgrad.py prints them).  Other builds ignore it. */
int rnvp_debug_set_trace(void* d_buf);

/* Tensor-core primitive self-test (tcgen05.mma kind::tf32, A in TMEM, B in shared memory):
 * D[128,N] = A[128,K] * B[N,K]^T on device buffers; passes = 1 (plain TF32) or 3 (split, fp32-grade). */
int rnvp_mma_selftest(const float* d_A, const float* d_B, float* d_D, int N, int K, int passes, void* stream);

/* Bootstrap metrics (rnvp_metrics.cu).  A bootstrap draw is given as per-row counts (bincount of the resampled row
 * indices), uint16, one row of counts per draw.  Precondition: within every draw, the counts of any 128 consecutive rows
 * of X (or of Y, tiles starting at row 0 of each) sum to at most 46340; otherwise d_median and d_mmd are NaN.
 *
 * rnvp_mmd_draws replaces mmd_calc over resample(X), resample(Y) (probaforms/metrics/mmd.py:8-21, :55-61) for n_draws
 * draws at once: d_median[b] = np.median of the pairwise distances of the drawn rows, d_mmd[b] = the RBF-kernel MMD with
 * gamma = 1 / (2 median^2).  d_X [n][D], d_Y [m][D] fp32; d_counts [n_draws][n+m] (X's counts first).  No n^2 buffer:
 * the workspace (rnvp_mmd_workspace_bytes) grows with n_draws only. */
int64_t rnvp_mmd_workspace_bytes(int64_t n, int64_t m, int D, int n_draws);
int rnvp_mmd_draws(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D,
                   const uint16_t* d_counts /* [n_draws][n+m] */, int n_draws,
                   double* d_median /* [n_draws] */, double* d_mmd /* [n_draws] */,
                   void* d_workspace, int64_t workspace_bytes, void* stream);
/* The same computation in stages, so that the pair tiles of one call can be split over n_shards devices (or streams)
 * and the host can merge the shards between stages (probaforms/metrics/mmd.py:8-21, :55-61; rnvp_mmd_draws is
 * begin, then hist_pass(p, 0, 1) + select(p) for p = 0, 1, 2, then sum_pass(0, 1) and finish).  Every shard has its own
 * workspace (rnvp_mmd_workspace_bytes) and all of them get the same leading arguments, as for rnvp_mmd_draws.
 *   begin      zero the workspace, per-draw count totals, selection state
 *   hist_pass  radix pass `pass` (0, 1, 2) over the pair tiles of shard `shard` (0 <= shard < n_shards); the shards of
 *              a call must run on devices with the same SM count
 *   merge      after each hist_pass: hist of every shard := the sum of the shards' hist (uint64), minval := their
 *              element-wise minimum (uint32; 0x7fffffff = none, so a signed int32 MIN gives the same result)
 *   select     pick the buckets of pass `pass`, zero hist; after pass 2, d_median and gamma (every shard, same result)
 *   sum_pass   the exponential sums of shard `shard`: its per-CTA rows of part, every other row stays +0.0
 *   merge      part of one workspace := the sum of the shards' part (fp64): exactly the single-shard values
 *   finish     d_mmd from that workspace
 * A shard with no pair tiles is valid and contributes zeros.  rnvp_mmd_layout gives the byte offsets and sizes of the
 * merged blocks within a workspace: offsets = { hist, hist bytes, minval, minval bytes, part, part bytes }. */
int rnvp_mmd_layout(int64_t n, int64_t m, int n_draws, int64_t* offsets /* [6] */);
int rnvp_mmd_begin(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts, int n_draws,
                   void* d_workspace, int64_t workspace_bytes, void* stream);
int rnvp_mmd_hist_pass(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts,
                       int n_draws, void* d_workspace, int64_t workspace_bytes, int pass, int shard, int n_shards,
                       void* stream);
int rnvp_mmd_select(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts, int n_draws,
                    void* d_workspace, int64_t workspace_bytes, int pass, double* d_median /* [n_draws] */, void* stream);
int rnvp_mmd_sum_pass(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts,
                      int n_draws, void* d_workspace, int64_t workspace_bytes, int shard, int n_shards, void* stream);
int rnvp_mmd_finish(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts, int n_draws,
                    void* d_workspace, int64_t workspace_bytes, double* d_mmd /* [n_draws] */, void* stream);
/* The moments behind X_boot.mean(axis=0) and np.cov(X_boot, rowvar=False) of frechet_distance
 * (probaforms/metrics/fd.py:40-47): d_sum[b] = sum_i c_bi x_i, d_outer[b] = sum_i c_bi x_i x_i^T in fp64
 * (fp32 products, fp64 combination; centre the rows first for an accurate covariance).  d_counts [n_draws][n]. */
int rnvp_boot_moments(const float* d_X, int64_t n, int D, const uint16_t* d_counts /* [n_draws][n] */, int n_draws,
                      double* d_sum /* [n_draws][D] */, double* d_outer /* [n_draws][D][D] */, void* stream);

/* Per-feature bootstrap metrics (rnvp_metrics1d.cu).  d_sorted [D][n+m] fp64 is each feature's pooled column [x; y]
 * sorted ascending, d_src [D][n+m] the row of each sorted position (rows < n are x's); d_counts [n_draws][n+m] uint16 as
 * above (x's counts first).  Requires n + m < 2^31.
 *
 * rnvp_rank_draws replaces, for every draw b and feature d, _ks1d, _cvm1d, _roc1d, _anderson1d
 * (probaforms/metrics/ks1d.py:11-30) and the histogram _kl1d, _js1d (div1d.py:6-44) over the drawn column:
 * d_stats[b][d][] = { ks_2samp statistic, cramervonmises_2samp statistic (NaN when n or m is 1), ROC AUC folded as
 * |auc - 0.5| + 0.5, anderson_ksamp's midrank A2kN (before the (A2kN - 1) / sigma standardisation), histogram KL,
 * histogram JS (bins, eps = 1e-5 / bins), the number of distinct drawn values }.  Workspace: rnvp_rank_workspace_bytes. */
#define RNVP_RANK_NSTAT 7
int64_t rnvp_rank_workspace_bytes(int D, int n_draws, int bins);
int rnvp_rank_draws(const double* d_sorted, const int32_t* d_src, int64_t n, int64_t m, int D,
                    const uint16_t* d_counts /* [n_draws][n+m] */, int n_draws, int bins, double eps,
                    double* d_stats /* [n_draws][D][RNVP_RANK_NSTAT] */, void* d_workspace, int64_t workspace_bytes,
                    void* stream);
/* The kernel sums behind compute_probs1d_kde (div1d.py:47-63): on the grid g = linspace(min, max, bins) of the drawn
 * pooled column, d_sums[b][d][0][k] = sum_{x rows} c_i exp(-(g_k - x_i)^2 / (2 h_x^2)) and d_sums[b][d][1][k] the same
 * over the y rows with h_y, in fp64.  Normalised to sum 1 they are the reference's p and q. */
int rnvp_kde_draws(const double* d_sorted, const int32_t* d_src, int64_t n, int64_t m, int D,
                   const uint16_t* d_counts /* [n_draws][n+m] */, int n_draws, int bins, double h_x, double h_y,
                   double* d_sums /* [n_draws][D][2][bins] */, void* stream);

/* ConditionalNormal (rnvp_cnormal.cu; probaforms/models/cnormal.py).  Net: model = Linear(Cd, h0), act, ..., act
 * (no final Linear), heads mu, log_sigma = Linear(h_last, D), out = Linear(D, D).  Parameters cross the boundary as one
 * flat fp32 buffer in Net.parameters() order: model.{2k}.weight [h_k, h_{k-1}], model.{2k}.bias, mu.weight, mu.bias,
 * log_sigma.weight, log_sigma.bias, out.weight [D, D], out.bias.  act: RNVP_ACT_TANH, _RELU or _SIGMOID (any other
 * activation string is ReLU upstream, cnormal.py:39-46).  Shapes: D <= 128, Cd <= 256, 1 to 4 hidden layers of width
 * <= 512 (RNVP_ESHAPE otherwise).  M is the caller-owned D x D inverse (W_out^T)^-1, row-major. */
enum { RNVP_ACT_SIGMOID = 3 };
typedef struct rnvp_cn_desc rnvp_cn_desc;
int rnvp_cn_desc_create(int D, int Cd, int n_hidden, const int* hidden, int act, int independent, rnvp_cn_desc** out);
void rnvp_cn_desc_destroy(rnvp_cn_desc* d);
int64_t rnvp_cn_param_count(const rnvp_cn_desc* d);
/* scratch bytes of rnvp_cn_grad / rnvp_cn_fit_epoch for batches of up to N rows (per-CTA gradient partials) */
int64_t rnvp_cn_workspace_bytes(const rnvp_cn_desc* d, int64_t N);
/* d_M = (W_out^T)^-1 by Gauss-Jordan with partial pivoting in fp32 (one CTA); *d_status = 1 on an exact-zero pivot,
 * untouched otherwise (the caller zeroes it) */
int rnvp_cn_inverse(const rnvp_cn_desc* d, const float* d_params, float* d_M, int* d_status, void* stream);
/* Net.forward for inference (cnormal.py:77-91): d_mu, d_sigma = exp(log_sigma), d_xtilde = mu + eps * sigma (then out()
 * in full-covariance mode), d_inv = (X - out.bias) M.  Every output may be NULL; d_inv needs d_X and d_M.  eps is d_eps
 * [N][D] when given (parity mode), else Philox keyed on (seed, row_offset + row, j) as in rnvp_sample. */
int rnvp_cn_forward(const rnvp_cn_desc* d, const float* d_params, const float* d_M, const float* d_X, const float* d_C,
                    int64_t N, uint64_t seed, int64_t row_offset, const float* d_eps, float* d_mu, float* d_sigma,
                    float* d_xtilde, float* d_inv, void* stream);
/* Exact log-density of the model's draws: d_logp[r] = log p(X[r] | C[r]) in fp64 (ConditionalNormal.log_prob_rows).
 * mu and log_sigma come from the fp32 net of rnvp_cn_forward (the same bits); then u = (x - out.bias) (W_out^T)^-1 in
 * full-covariance mode (u = x in independent mode) and
 *   log p = -1/2 sum_d ((u_d - mu_d) / sigma_d)^2 - sum_d log_sigma_d - (D/2) log 2 pi - log|det W_out|,
 * summed in fp64, log sigma taken from the head directly.  Full mode first factors W_out^T in fp64 with the partial
 * pivoting of rnvp_cn_inverse: log|det W_out| = sum of log|pivot|, and the fp64 inverse, into d_workspace (1 + D * D
 * doubles); an exact-zero pivot sets *d_status = 1 (the caller zeroes it) and leaves d_logp untouched.  Independent
 * mode needs neither d_workspace nor d_status. */
int rnvp_cn_log_prob(const rnvp_cn_desc* d, const float* d_params, const float* d_X, const float* d_C, int64_t N,
                     double* d_logp, double* d_workspace, int* d_status, void* stream);
/* loss (cnormal.py:140-151) and its gradient on the N rows X[idx[r]], C[idx[r]] (d_idx may be NULL): d_gflat [P] in
 * the flat layout (zeros for out.* in independent mode, where the loss does not depend on them), *d_loss */
int rnvp_cn_grad(const rnvp_cn_desc* d, const float* d_params, const float* d_M, const float* d_X, const float* d_C,
                 const int64_t* d_idx, int64_t N, float* d_gflat, float* d_loss, void* d_workspace,
                 int64_t workspace_bytes, void* stream);
/* One epoch of ConditionalNormal.fit (cnormal.py:193-209) as one call: for every consecutive batch_size slice of d_perm
 * (last partial batch kept), loss + gradient + torch.optim.Adam step (step count step0 + 1, ...; out.* skipped in
 * independent mode), loss to d_losses[s], and in full mode d_M refreshed for the next step.  A batch of at most the
 * kernel's tile (64 rows for small nets) is one launch.  If a refreshed W_out has an exact-zero pivot, *d_status =
 * (fit step index of the next step) + 1 and every later step of this and later calls with the same d_status is a
 * no-op.  Workspace: rnvp_cn_workspace_bytes(d, batch_size). */
int rnvp_cn_fit_epoch(const rnvp_cn_desc* d, float* d_params, float* d_exp_avg, float* d_exp_avg_sq, float* d_M,
                      const float* d_X, const float* d_C, const int64_t* d_perm, int64_t n, int64_t batch_size,
                      double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step0,
                      float* d_losses, int* d_status, void* d_workspace, int64_t workspace_bytes, void* stream);
/* Host only: advance a torch CPU generator state (Generator.get_state() bytes, 5056) exactly as torch.randn(numel) in
 * float32 does, for numel >= 16 (numel 32-bit draws, plus 16 when numel % 16 != 0); smaller numel: RNVP_EINVAL. */
int rnvp_cn_rng_advance(uint8_t* state, int64_t state_bytes, int64_t numel);

/* CVAE (rnvp_cvae.cu; probaforms/models/cvae.py).  Encoder: model = Linear(D + Cd, h0), act, ..., act, heads mu,
 * log_sigma = Linear(h_last, latent); Decoder: model = Linear(latent + Cd, h0), act, ..., act, Linear(h_last, D)
 * (cvae.py:14-110).  Parameters cross the boundary as one flat fp32 buffer in the order of the reference's Adam
 * (cvae.py:173): encoder.model.{2k}.weight [h_k, h_{k-1}], encoder.model.{2k}.bias, encoder.mu.weight, .bias,
 * encoder.log_sigma.weight, .bias, then decoder.model.{2k}.weight, .bias and decoder.model.{2 nh}.weight [D, h_last],
 * .bias.  act: RNVP_ACT_TANH or _RELU (every other activation string is ReLU upstream, cvae.py:27-32).  Cd may be 0 (the
 * reference's C=None, cvae.py:158-161); d_C may then be NULL.  Shapes: D <= 128, Cd <= 256, latent <= 128, 1 to 4
 * hidden layers of width <= 512 (RNVP_ESHAPE otherwise).  eps buffers are [N][latent], indexed by batch position. */
typedef struct rnvp_cv_desc rnvp_cv_desc;
int rnvp_cv_desc_create(int D, int Cd, int latent, int n_hidden, const int* hidden, int act, rnvp_cv_desc** out);
void rnvp_cv_desc_destroy(rnvp_cv_desc* d);
int64_t rnvp_cv_param_count(const rnvp_cv_desc* d);
/* scratch bytes for gradient batches of up to batch_rows rows (per-CTA gradient partials) and loss passes of up to
 * loss_rows rows (per-CTA loss partials) */
int64_t rnvp_cv_workspace_bytes(const rnvp_cv_desc* d, int64_t batch_rows, int64_t loss_rows);
/* Encoder.forward for inference (cvae.py:38-62): d_mu, d_log_sigma [N][latent] of the rows [X | C] */
int rnvp_cv_encode(const rnvp_cv_desc* d, const float* d_params, const float* d_X, const float* d_C, int64_t N,
                   float* d_mu, float* d_log_sigma, void* stream);
/* Decoder.forward for inference (cvae.py:89-110): d_x [N][D] of the rows [Z | C]; Z is d_Z [N][latent] when given
 * (parity mode), else Philox normals keyed on (seed, row_offset + row, j) as in rnvp_sample (replaces the CPU
 * torch.normal of sample, cvae.py:283-290) */
int rnvp_cv_decode(const rnvp_cv_desc* d, const float* d_params, const float* d_Z, const float* d_C, int64_t N,
                   uint64_t seed, int64_t row_offset, float* d_x, void* stream);
/* compute_loss (cvae.py:190-199) and its gradient on the N rows X[idx[r]], C[idx[r]] (d_idx may be NULL) with the
 * caller's eps (sample_z, cvae.py:181-183): d_gflat [P] in the flat layout, *d_loss (may be NULL).
 * Workspace: rnvp_cv_workspace_bytes(d, N, 0). */
int rnvp_cv_grad(const rnvp_cv_desc* d, const float* d_params, const float* d_X, const float* d_C,
                 const int64_t* d_idx, const float* d_eps, int64_t N, double kl_weight, float* d_gflat, float* d_loss,
                 void* d_workspace, int64_t workspace_bytes, void* stream);
/* compute_loss alone (forward only) into *d_loss.  Workspace: rnvp_cv_workspace_bytes(d, 0, N). */
int rnvp_cv_loss(const rnvp_cv_desc* d, const float* d_params, const float* d_X, const float* d_C,
                 const int64_t* d_idx, const float* d_eps, int64_t N, double kl_weight, float* d_loss,
                 void* d_workspace, int64_t workspace_bytes, void* stream);
/* One epoch of CVAE.fit (cvae.py:232-255) as one call: for every consecutive batch_size slice of d_perm (last partial
 * batch kept), loss + gradient + torch.optim.Adam step (step count step0 + 1, ...), then compute_loss over all n rows
 * in dataset order into *d_loss.  Noise: d_noise holds every step's [nb][latent] eps in step order followed by the
 * [n][latent] eps of the epoch loss; when NULL, Philox keyed on (seed, position in the epoch order, j) for the steps and
 * (seed, n + row, j) for the epoch loss.  A batch of at most the kernel's tile (64 rows for small nets) is one launch.
 * Workspace: rnvp_cv_workspace_bytes(d, min(batch_size, n), n). */
int rnvp_cv_fit_epoch(const rnvp_cv_desc* d, float* d_params, float* d_exp_avg, float* d_exp_avg_sq, const float* d_X,
                      const float* d_C, const int64_t* d_perm, int64_t n, int64_t batch_size, double lr, double beta1,
                      double beta2, double eps, double weight_decay, double kl_weight, int64_t step0,
                      const float* d_noise, uint64_t seed, float* d_loss, void* d_workspace, int64_t workspace_bytes,
                      void* stream);

/* ConditionalWGAN (rnvp_wgan.cu; probaforms/models/wgan.py).  Generator: model = Linear(latent + Cd, g_h0), act, ...,
 * act, Linear(g_h_last, D); Discriminator (the critic): model = Linear(D + Cd, d_h0), act, ..., act, Linear(d_h_last, 1)
 * (wgan.py:12-107).  Parameters cross the boundary as one flat fp32 buffer: generator.parameters() (model.{2k}.weight
 * [h_k, h_{k-1}], model.{2k}.bias, ..., model.{2 nh}.weight, .bias), then discriminator.parameters() in the same form.
 * Each net has its own hidden tuple and act (RNVP_ACT_TANH or _RELU: every other activation string is ReLU upstream,
 * wgan.py:26-31).  Cd may be 0 (the reference's C=None); d_C may then be NULL.  Shapes: D <= 128, Cd <= 256,
 * latent <= 128, 1 to 4 hidden layers of width <= 512 per net (RNVP_ESHAPE otherwise).  z buffers are [N][latent],
 * indexed by batch position. */
typedef struct rnvp_wg_desc rnvp_wg_desc;
int rnvp_wg_desc_create(int D, int Cd, int latent, int g_hidden_n, const int* g_hidden, int g_act, int d_hidden_n,
                        const int* d_hidden, int d_act, rnvp_wg_desc** out);
void rnvp_wg_desc_destroy(rnvp_wg_desc* d);
/* parameters of the generator (net 0), of the discriminator (net 1) or of both (any other net) */
int64_t rnvp_wg_param_count(const rnvp_wg_desc* d, int net);
/* scratch bytes for gradient batches of up to batch_rows rows (per-CTA gradient partials) and loss passes of up to
 * loss_rows rows (per-CTA score sums) */
int64_t rnvp_wg_workspace_bytes(const rnvp_wg_desc* d, int64_t batch_rows, int64_t loss_rows);
/* Generator.forward for inference (wgan.py:38-58): d_x [N][D] of the rows [Z | C]; Z is d_Z [N][latent] when given
 * (parity mode), else Philox normals keyed on (seed, row_offset + row, j) as in rnvp_sample (replaces the CPU
 * torch.normal of sample, wgan.py:314-318) */
int rnvp_wg_generate(const rnvp_wg_desc* d, const float* d_params, const float* d_Z, const float* d_C, int64_t N,
                     uint64_t seed, int64_t row_offset, float* d_x, void* stream);
/* Discriminator.forward for inference (wgan.py:86-107): d_score [N] of the rows [X | C] */
int rnvp_wg_critic(const rnvp_wg_desc* d, const float* d_params, const float* d_X, const float* d_C, int64_t N,
                   float* d_score, void* stream);
/* One step's loss and gradient on the N rows X[idx[r]], C[idx[r]] (d_idx may be NULL) with the caller's latent z, no
 * optimizer update: a critic step (generator_step 0: loss_disc = -mean(D([x|c])) + mean(D([G([z|c])|c])), gradient of
 * the discriminator's parameters) or a generator step (1: loss_gen = -mean(D([G([z|c])|c])), gradient of the
 * generator's) (wgan.py:225-273).  d_gflat [P] in the flat layout, zero over the other net; *d_loss (may be NULL).
 * Workspace: rnvp_wg_workspace_bytes(d, N, 0). */
int rnvp_wg_grad(const rnvp_wg_desc* d, const float* d_params, const float* d_X, const float* d_C,
                 const int64_t* d_idx, const float* d_z, int64_t N, int generator_step, float* d_gflat, float* d_loss,
                 void* d_workspace, int64_t workspace_bytes, void* stream);
/* The epoch losses (wgan.py:280-293) of the N rows: *d_gen_loss = -mean(D([G([z|c])|c])), *d_disc_loss =
 * mean(D([x|c])) + *d_gen_loss.  Workspace: rnvp_wg_workspace_bytes(d, 0, N). */
int rnvp_wg_loss(const rnvp_wg_desc* d, const float* d_params, const float* d_X, const float* d_C,
                 const int64_t* d_idx, const float* d_z, int64_t N, float* d_gen_loss, float* d_disc_loss,
                 void* d_workspace, int64_t workspace_bytes, void* stream);
/* One epoch of ConditionalWGAN.fit (wgan.py:222-295) as one call: for every consecutive batch_size slice of d_perm
 * (last partial batch kept), fit step i = step0, step0 + 1, ... (counted over the whole fit) is a generator step when
 * i % n_critic == 0 and a critic step otherwise; each runs torch.optim.RMSprop (lr, alpha, eps, weight_decay; momentum
 * 0, not centred) on its own net with d_square_avg [P] as the state, and a critic step then clamps every discriminator
 * parameter to [-clip, clip].  Then the epoch losses over all n rows in dataset order into *d_gen_loss, *d_disc_loss.
 * Noise: d_noise holds every step's [nb][latent] z in step order followed by the [n][latent] z of the epoch losses;
 * when NULL, Philox keyed on (seed, position in the epoch order, j) for the steps and (seed, n + row, j) for the epoch
 * losses.  A batch of at most the kernel's tile (64 rows for small nets) is one launch.
 * Workspace: rnvp_wg_workspace_bytes(d, min(batch_size, n), n). */
int rnvp_wg_fit_epoch(const rnvp_wg_desc* d, float* d_params, float* d_square_avg, const float* d_X, const float* d_C,
                      const int64_t* d_perm, int64_t n, int64_t batch_size, int64_t n_critic, int64_t step0, double lr,
                      double alpha, double eps, double weight_decay, double clip, const float* d_noise, uint64_t seed,
                      float* d_gen_loss, float* d_disc_loss, void* d_workspace, int64_t workspace_bytes,
                      void* stream);

/* Predictive summaries (rnvp_summary.cu; probaforms_b200/predictive.py).  Per cell c < cells of the k draws laid out
 * d_draws[j * cells + c] (cell = row * D + feature):
 *   d_mean, d_std (ddof = 0) in fp64 with a fixed summation order; the nq quantiles of numpy's default 'linear' method,
 *   equal bit for bit to np.quantile(draws, q, axis=0) of the float32 draws (NaN for every quantile of a cell with a
 *   NaN draw); with d_y [cells]: d_crps = (1/k) sum_j |x_j - y| - (1/(2 k^2)) sum_i sum_j |x_i - x_j| (NaN for a NaN y)
 *   and d_rank = #{j : x_j < y}.
 * Output pointers may be NULL (skipped); d_crps / d_rank need d_y.  q is a HOST array of nq <= 32 values in [0, 1].
 * Quantile plane i is written at d_quant + i * q_stride (q_stride >= cells), so row blocks can write straight into
 * full-size outputs.  RNVP_EINVAL for k < 1 or k > RNVP_SUMMARY_MAX_DRAWS and the other bad arguments. */
#define RNVP_SUMMARY_MAX_DRAWS 8192
#define RNVP_SUMMARY_MAX_QUANTILES 32
int rnvp_draw_summary(const float* d_draws, int64_t k, int64_t cells, const double* q, int nq, const float* d_y,
                      double* d_mean, double* d_std, double* d_quant, int64_t q_stride, double* d_crps,
                      int32_t* d_rank, void* stream);

/* Joint scores of k draws per row (rnvp_summary.cu; probaforms_b200/predictive.py predictive_joint).  The draws of a
 * block of rows are laid out d_draws[(j * rows + r) * D + d] (draw j, row r, feature d), 1 <= D <= RNVP_JOINT_MAX_D.
 * Per row r:
 *   d_mean [rows, D] (required): the fp64 mean of the draws, summed in a fixed order;
 *   d_cov [rows, D, D] (NULL: skipped): sum_j (x_j - mean)(x_j - mean)^T / k, both triangles;
 *   with d_y [rows, D]: d_energy [rows] = (1/k) sum_j ||x_j - y|| - (1/(2 k^2)) sum_i sum_j ||x_i - x_j|| (Euclidean)
 *   and d_variogram [rows] = sum_{d<e} (|y_d - y_e|^p - (1/k) sum_j |x_jd - x_je|^p)^2 (NULL: skipped).
 * A row with a non-finite draw gives NaN cov, energy and variogram; a NaN in y gives NaN energy and variogram.
 * d_energy needs a device workspace of rnvp_draw_joint_workspace_bytes(k, rows, D) bytes (rows x tile pairs doubles;
 * -1 for bad arguments).  Results are bitwise repeatable and do not depend on how rows are split into calls.
 * RNVP_EINVAL for k outside [1, RNVP_SUMMARY_MAX_DRAWS], D outside [1, RNVP_JOINT_MAX_D], p not finite and > 0, and
 * the other bad arguments. */
#define RNVP_JOINT_MAX_D 128
int64_t rnvp_draw_joint_workspace_bytes(int64_t k, int64_t rows, int D);
int rnvp_draw_joint(const float* d_draws, int64_t k, int64_t rows, int D, const float* d_y, double p, double* d_mean,
                    double* d_cov, double* d_energy, double* d_variogram, void* d_workspace, int64_t workspace_bytes,
                    void* stream);

/* Predictive log scores of k draws per row (rnvp_density.cu; probaforms_b200/predictive.py predictive_density).  The
 * draws are laid out as for rnvp_draw_joint, 1 <= D <= RNVP_JOINT_MAX_D and D < k <= RNVP_SUMMARY_MAX_DRAWS; d_y
 * [rows, D] is required.  Per row r, with the draws x_j promoted to fp64, S their covariance (ddof = 1, a centred
 * two-pass sum) and S = L L^T:
 *   d_log_score [rows] = -(logsumexp_j(-1/2 ||(f L)^-1 (y - x_j)||^2) - log k - sum_i log(f L_ii) - (D/2) log 2 pi),
 *     the negative log of the Gaussian KDE with bandwidth matrix f^2 S (scipy's gaussian_kde with factor f), with a
 *     max-shifted logsumexp;
 *   d_dss [rows] = 2 sum_i log L_ii + ||L^-1 (y - mean)||^2, the Dawid-Sebastiani score;
 *   d_marginal [rows, D] (NULL: skipped) = the 1-D KDE log score of each feature, bandwidth factor1 * sigma_d with
 *     sigma_d^2 = S_dd.
 * Rules: a row with a non-finite draw or a non-finite y gives NaN log score, DSS and marginals.  A Cholesky pivot
 * L_ii^2 <= 1e-12 S_ii (this covers a zero-variance feature) makes S degenerate: NaN log score and DSS, while the
 * marginals stay defined.  A constant feature (S_dd = 0) gives a NaN marginal.  These differ from scipy, which raises
 * only when LAPACK's factorisation fails.  No workspace.  Results are bitwise repeatable and do not depend on how rows
 * are split into calls.  RNVP_EINVAL for D outside [1, RNVP_JOINT_MAX_D], k outside (D, RNVP_SUMMARY_MAX_DRAWS], a
 * factor (or, with d_marginal, factor1) that is not finite and > 0, and the other bad arguments. */
int rnvp_draw_density(const float* d_draws, int64_t k, int64_t rows, int D, const float* d_y, double factor,
                      double factor1, double* d_log_score, double* d_dss, double* d_marginal, void* stream);

const char* rnvp_last_error(void);
int rnvp_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RNVP_H */
