/*
 * ssac_b200.h -- C ABI of libssac_b200.so: the off-policy update step of jakegrigsby/super_sac as
 * hand-written sm_100a CUDA.  The reference is pure Python/PyTorch and has no FFI of its own; each
 * entry point below replaces the ATen call sequence of the cited reference lines (paths relative to the
 * reference root).  INTEGRATION.md shows the ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no C++ / torch types cross the boundary.
 *   - every pointer named *_dev / documented "device" is a CUDA device pointer owned by the caller
 *     (PyTorch owns all tensors); the library never frees or allocates caller memory on the hot path.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises.
 *     Every call is CUDA-graph capturable (no malloc, no sync, pointer-stable arguments); values that
 *     change between replays (Adam step, PopArt state, Philox offset, log_alpha) live in device memory.
 *   - return 0 on success, else a cudaError_t or a negative SSAC_E_* code; ssac_last_error() gives the
 *     message of the last failure on the calling thread.  No exceptions cross the ABI.
 *   - hyper-parameters the reference keeps as Python floats (lr, betas, eps, tau, ...) cross as double so that
 *     derived constants (1-beta2, 1-tau, bias corrections) round exactly like the reference's.
 *   - all floating point is IEEE fp32 (the reference runs true-fp32 SGEMM, SURVEY F12); replay / gather /
 *     augmentation / segment-tree entry points are bit-exact integer, byte or float64 work.
 *   - matrices are row-major; "ld" = elements between consecutive rows; "gs" = elements between groups.
 */
#ifndef SSAC_B200_H
#define SSAC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSAC_E_BADARG (-1)
#define SSAC_E_UNSUPPORTED (-2)
#define SSAC_E_ARCH (-3)

/* ---- library ------------------------------------------------------------------------------------- */
const char* ssac_last_error(void);
int ssac_version(void);
/* 0 iff `device` is an sm_100 part (the library carries sm_100a SASS only: no fallback). */
int ssac_device_check(int device);

/* ---- target networks: learning_utils.py:160-167 (soft_update / hard_update), main.py:409-414 ------ */
/* target <- target*(1-tau) + source*tau, three separately rounded fp32 ops: bit-exact with the reference. */
int ssac_polyak(float* target_dev, const float* source_dev, int64_t n, double tau, void* stream);
/* Same over a table of tensors (user encoders are arbitrary nn.Modules): table_dev = n_tensors x
 * {uint64 target_ptr, uint64 source_ptr, uint64 numel}; total_chunks = sum ceil(numel/chunk). */
int ssac_polyak_multi(const uint64_t* table_dev, int n_tensors, int64_t max_numel, double tau, void* stream);

/* ---- optimiser: torch.optim.Adam as configured in main.py:188-239 (coupled L2, no amsgrad) -------- */
/* ctl_dev: int32[2] = {step, blocks_done}; the kernel reads step, uses t = step+1 for the bias
 * corrections and the last block to finish stores step+1 (graph replays advance it).
 * gnorm_sq_dev (nullable): if given with max_norm > 0, grads are scaled by
 * min(1, max_norm/(sqrt(*gnorm_sq_dev)+1e-6)) (torch.nn.utils.clip_grad_norm_, learning.py:122-128) and,
 * if write_back_grad, the scaled gradient is stored to g_dev like clip_grad_norm_ does. */
int ssac_adam_step(float* p_dev, float* g_dev, float* m_dev, float* v_dev, int64_t n, int32_t* ctl_dev,
                   double lr, double beta1, double beta2, double eps, double weight_decay,
                   const float* gnorm_sq_dev, double max_norm, int write_back_grad, void* stream);
/* Adam followed by the Polyak update of the matching target parameters in one pass (36 B/param). */
int ssac_adam_polyak_step(float* p_dev, float* g_dev, float* m_dev, float* v_dev, float* target_dev, int64_t n,
                          int32_t* ctl_dev, double lr, double beta1, double beta2, double eps, double weight_decay,
                          const float* gnorm_sq_dev, double max_norm, int write_back_grad, double tau, void* stream);
/* x_dev[i] = *scale_dev * x_dev[i]: the annealed exploration-noise scale of learning_utils.py:48-59 kept in device memory
 * (GaussianExplorationNoise.scale_dev), so that a captured update follows it from replay to replay. */
int ssac_scale_by_dev(float* x_dev, int64_t n, const float* scale_dev, void* stream);
/* out_dev[0] (+)= sum x^2  (global grad norm for clipping / get_grad_norm, learning_utils.py:95-106). */
int ssac_sumsq(const float* x_dev, int64_t n, float* out_dev, int accumulate, void* stream);

/* ---- random draws: replay.py:122 (indices), agent.py:29 (REDQ subset), Normal sampling, ------------
 * learning_utils.py:49 (TD3 noise), augmentations.py:180-181,227-231 (shifts).  Philox4x32-10.
 * rng_dev: uint64[4] = {seed, offset, blocks_done, reserved}; the kernel's last block advances offset so that
 * graph replays draw fresh numbers.  Any output may be NULL.
 *   idx_dev     int64[n_idx]            uniform in [0, n_filled); n_filled_dev (nullable device int64[1]) overrides
 *                                       n_filled so that a captured graph follows a growing buffer
 *   normal_dev  float[n_normal]         N(0,1)
 *   subset_dev  int32[n_subsets*M]      n_subsets independent M-subsets of {0..N-1} (without replacement)
 *   shift_dev   int32[n_shift]          uniform in [0, shift_range)
 *   zero_dev    float[n_zero]           set to 0 (the update's scalar-log / loss accumulators ride along instead of
 *                                       costing a memset launch of their own)                            */
int ssac_rng_fill(uint64_t* rng_dev, int64_t* idx_dev, int64_t n_idx, int64_t n_filled, const int64_t* n_filled_dev,
                  float* normal_dev, int64_t n_normal, int32_t* subset_dev, int n_subsets, int N, int M, int32_t* shift_dev,
                  int64_t n_shift, int shift_range, float* zero_dev, int64_t n_zero, void* stream);

/* ---- replay gather: replay.py:66-84 + learning_utils.py:186-197 (H2D + .float()) ------------------ */
/* For each of n_arrays arrays: dst[b, :] = src[idx[b], :].  row_elems[k] elements per row;
 * mode[k]: 0 = f32 -> f32 copy, 1 = u8 -> f32 cast, 2 = raw bytes (row_elems = bytes per row).
 * dst_ld[k] = elements between dst rows (lets a gather write straight into a column block of a wider
 * matrix such as cat(s, a)).  srcs/dsts/... are HOST arrays of n_arrays (<= 16) entries. */
int ssac_gather_rows(const void* const* srcs_dev, void* const* dsts_dev, const int64_t* row_elems,
                     const int64_t* dst_ld, const int32_t* mode, int n_arrays, const int64_t* idx_dev, int B,
                     void* stream);
/* Ring write of one pushed transition (replay.py:48-61): the host packs every field (s, s1, action, reward, done, tree
 * index / priority, fill level) into ONE pinned staging buffer that crosses PCIe with a single copy; this kernel then
 * scatters field k (nbytes[k] bytes at staging_dev + src_off[k]) to dsts_dev[k].  Host arrays of n_fields (<= 16). */
int ssac_scatter_fields(const void* staging_dev, void* const* dsts_dev, const int64_t* nbytes, const int64_t* src_off,
                        int n_fields, void* stream);
/* The whole single-transition push in one call: H2D copy of the pinned staging row (row_bytes) into staging_dev, the field
 * scatter of ssac_scatter_fields, and -- when sum_tree is given -- the PER leaf write + ancestor update of ssac_tree_set
 * for the leaf index (int64 at staging + tree_idx_off) and priority (float64 at staging + tree_val_off).  `slot`
 * (0..63) names the pinned row: the call records an event behind its copy, and ssac_push_row_wait(slot) blocks the host
 * until that copy has completed (call it before refilling the pinned row); wait_slot >= 0 does that wait for another
 * slot (the one the host fills next) at the end of this call, saving the separate call.  wait_event (nullable
 * cudaEvent_t): the stream waits for it before anything else (an update in flight that may still read the ring slot). */
int ssac_push_row(const void* host_row_pinned, void* staging_dev, int64_t row_bytes, int slot, void* const* dsts_dev,
                  const int64_t* nbytes, const int64_t* src_off, int n_fields, double* sum_tree_dev, double* min_tree_dev,
                  int64_t capacity, int64_t tree_idx_off, int64_t tree_val_off, int wait_slot, void* wait_event, void* stream);
int ssac_push_row_wait(int slot);
/* ssac_push_row with a list of PER leaf writes instead of one (prioritised frame-deduplicated n-step ring: a push may evict
 * transitions -- their leaves get sum 0, min +inf -- and add one at max_priority ** alpha).  The staging row holds, at
 * leaves_off, int64 leaf[n_leaves], then float64 sum value[n_leaves], then float64 min value[n_leaves] (1..256 writes); they
 * are applied in order (the last write of a leaf wins), each with the ancestor update of ssac_push_row, in the same launch
 * as the field scatter. */
int ssac_push_row_leaves(const void* host_row_pinned, void* staging_dev, int64_t row_bytes, int slot, void* const* dsts_dev,
                         const int64_t* nbytes, const int64_t* src_off, int n_fields, double* sum_tree_dev, double* min_tree_dev,
                         int64_t capacity, int64_t leaves_off, int n_leaves, int wait_slot, void* wait_event, void* stream);
/* Fused pixel gather + DrQ / DrQv2 random shift + uint8 -> fp32 + aug_mix: augmentations.py:165-269,
 * learning_utils.py:193-206.   src u8 [capacity, C, H, W] -> dst f32 [B, C, H, W].
 * pad_mode 0: no shift, 1: replicate (DrQv2 integer crop), 2: reflect (DrQ v1), 3: RAD (augmentations.py:129-162:
 * cv2 bilinear upscale by `pad` (= crop) pixels per axis, then the H x W window at offset shift; same fp32
 * arithmetic as cv2.resize(INTER_LINEAR) on float32 data, bit-exact on frame stacks of more than 4 channels).
 * shift_dev int32 [B,2] = (x, y) with 0 <= shift <= 2*pad (v2) / < 2*pad (v1) / < crop (RAD).  Rows b < aug_rows are
 * augmented, the rest are a plain cast.  noise_dev (nullable) f32 [B,C,H,W] is added before the clamp to
 * [0,255] (DrqAug noise=True). */
int ssac_gather_aug_u8(const uint8_t* src_dev, float* dst_dev, const int64_t* idx_dev, const int32_t* shift_dev,
                       const float* noise_dev, int B, int C, int H, int W, int pad, int pad_mode, int aug_rows,
                       void* stream);

/* The same gather over a ring of SINGLE FRAMES (frame-deduplicated layout, SURVEY 8f N2): an observation is C consecutive
 * planes starting at frame first_frame_dev[b] (a monotonically increasing frame counter; taken modulo ring_frames), so a
 * frame stack s_t = [f_{t-k+1} .. f_t] and its successor s_{t+1} share k-1 stored frames and every frame is stored once
 * (reference layout: s and s1 stacks side by side, replay.py:10-61: 2k copies).  pad_mode 0..2. */
int ssac_gather_aug_u8_ring(const uint8_t* frames_dev, float* dst_dev, const int64_t* first_frame_dev,
                            int64_t planes_per_frame, int64_t ring_frames, const int32_t* shift_dev, const float* noise_dev,
                            int B, int C, int H, int W, int pad, int pad_mode, int aug_rows, void* stream);
/* On-the-fly n-step transitions (main.py:353-365, learning_utils.py:139-151 moved into the sampler).  The ring holds
 * one-step transitions in time order; valid_ring_dev (int64[cap], a FIFO whose oldest entry sits at scalars_dev[1] =
 * v_tail; scalars_dev[0] = number of entries, the `n_filled` the index draw uses) lists the slots whose n-step window
 * lies inside one episode.  For position j_dev[b]: idx_start = that slot, idx_last = slot of step t+n-1 (its next state
 * and done flag are the transition's), R = r_t + gamma r_{t+1} + ... accumulated left to right like the reference's loop:
 * in float64 over reward64_dev, or in float32 over reward32_dev (float32(gamma^i) * r_i: what NumPy does with np.float32
 * rewards); gamma_pows_dev float64[n_step] = gamma**i.  first_frame_dev (nullable, frame-deduplicated layout): frame
 * counter of each step's state stack -> frame_s / frame_s1 for ssac_gather_aug_u8_ring. */
int ssac_nstep_resolve(const int64_t* j_dev, int B, const int64_t* valid_ring_dev, const int64_t* scalars_dev, int64_t cap,
                       int n_step, const double* reward64_dev, const float* reward32_dev, const double* gamma_pows_dev,
                       const int64_t* first_frame_dev, int64_t* idx_start_dev, int64_t* idx_last_dev, float* R_dev,
                       int64_t* frame_s_dev, int64_t* frame_s1_dev, void* stream);

/* ---- prioritised replay: replay.py:163-190, :207-353 (float64 sum / min segment trees) ------------ */
/* tree layout identical to the reference: value[2*capacity], root at 1, leaves at capacity + i. */
int ssac_tree_set(double* sum_tree_dev, double* min_tree_dev, int64_t capacity, const int64_t* idx_dev,
                  const double* val_dev, int64_t n, void* stream);
/* idx_out[b] = find_prefixsum_idx(u[b] * sum(0, n_filled-1)); weights as replay.py:173-176. */
int ssac_tree_sample(const double* sum_tree_dev, const double* min_tree_dev, int64_t capacity, int64_t n_filled,
                     const double* u01_dev, int B, double beta, int64_t* idx_out_dev, double* weight_out_dev,
                     void* stream);
/* Prioritised replay over the frame-deduplicated n-step ring (SURVEY 8f N2).  A transition's leaf is its slot in the FIFO
 * of valid starts, v mod ring_size (v = running count of starts); the trees have capacity >= ring_size leaves.
 * scalars_dev = the ring's device int64 {n_valid, v_tail % ring_size, v_tail}; the live leaves are the circular range
 * [v_tail, v_tail + n_valid) mod ring_size, every other leaf holds (sum 0, min +inf).
 * ssac_tree_set_live: ssac_tree_set (n <= 1024, last write wins) that drops every id whose slot is not live when the
 * kernel runs (evicted since it was sampled and not yet reused): a dead leaf never gets priority back. */
int ssac_tree_set_live(double* sum_tree_dev, double* min_tree_dev, int64_t capacity, int64_t ring_size, const int64_t* scalars_dev,
                       const int64_t* idx_dev, const double* val_dev, int64_t n, void* stream);
/* Proportional draw + importance weights + the n-step resolve of ssac_nstep_resolve, in one launch (B <= 1024).
 *   v_tail == 0 (no start evicted yet): exactly ssac_tree_sample with n_filled = n_valid (mass u * sum(0, n_valid-1)).
 *   v_tail > 0: mass u * root sum (every live transition can be drawn); weights of replay.py:173-176 with N = n_valid and
 *     p_min = min root / sum root.
 * A descent that float64 rounding lands on a dead leaf is moved to the live leaf with the largest index below it, or, when
 * no live leaf lies below it, to the oldest live leaf: no dead slot is ever returned.  slot_out = leaf ids (what
 * ssac_tree_set_live takes), j_out (nullable) = FIFO positions (slot - v_tail) mod ring_size, weight_out (nullable)
 * float64; the remaining arguments and outputs are those of ssac_nstep_resolve. */
int ssac_nstep_tree_sample(const double* sum_tree_dev, const double* min_tree_dev, int64_t capacity, int64_t ring_size,
                           const int64_t* scalars_dev, const double* u01_dev, int B, double beta, int64_t* slot_out_dev,
                           int64_t* j_out_dev, double* weight_out_dev, const int64_t* valid_ring_dev, int n_step,
                           const double* reward64_dev, const float* reward32_dev, const double* gamma_pows_dev,
                           const int64_t* first_frame_dev, int64_t* idx_start_dev, int64_t* idx_last_dev, float* R_dev,
                           int64_t* frame_s_dev, int64_t* frame_s1_dev, void* stream);

/* ---- ensemble MLPs: agent.py:13-40 (Critic), nets/mlps.py:11-41,78-93,113-129 --------------------- */
/* G independent 3-Linear ReLU MLPs  D -> H -> H -> O.  Parameters: W1 [nets,H,D] b1 [nets,H] W2 [nets,H,H]
 * b2 [nets,H] W3 [nets,O,H] b3 [nets,O] (nn.Linear layout).  Group g uses net net_index_dev[g] (device
 * int32, e.g. the REDQ subset) or net g when NULL.  Input x_dev: row-major [.,B,D] with row stride ldx and
 * group stride x_gs (0 = every group reads the same batch).  Outputs h1/h2 [G,B,H] (nullable: not saved),
 * y [G,B,O].  impl: 0 = library default (ssac_set_default_mlp_impl), 1 = fp32 FFMA tiles, 2 = tcgen05 tensor cores
 * with 3xTF32 operand splitting (fp32-accurate: hi*hi + hi*lo + lo*hi, fp32 accumulation in TMEM), 3 = the row-local
 * CUDA-core kernel below (forward-only: keep_hidden == 0, shared input x_gs == 0, ssac_rows_supported shapes). */
int ssac_default_mlp_impl(void);
int ssac_set_default_mlp_impl(int impl);
/* impl 2 stages operands with TMA (cp.async.bulk.tensor) when their pitch allows; 0 forces the register-staged path
 * (kept for cross-checking the two staging paths against each other). */
int ssac_set_tma_enabled(int on);
/* ssac_mlp_backward runs its weight-gradient branch (gW3, gW2, and gW1 when dx is also wanted) on an internal side
 * stream, forked from / joined into `stream` with events (graph edges under stream capture); 0 serialises everything
 * on `stream`.  Results are identical either way.  Default 1. */
int ssac_set_overlap(int on);
int ssac_get_overlap(void);
/* Programmatic dependent launch for the kernels of the update's critical path (replay gather, single-kernel forward, TD
 * target, dz2, dz1 GEMM, gW1): each is launched so that its set-up (TMEM allocation, barrier init, parameter loads)
 * overlaps the tail of its predecessor in the stream; `griddepcontrol.wait` guards everything an earlier kernel
 * produced.  0 = plain stream-ordered launches.  Results are identical.  Default 1. */
int ssac_set_pdl(int on);
int ssac_get_pdl(void);
/* impl 2, 2 x 256-class networks (H in 32..256 and a multiple of 16, first-layer width <= 64, O <= 32): the whole forward
 * (three layers + head epilogue) runs as ONE kernel that keeps the activations in tensor / shared memory.  h1 / h2 are
 * then written only when keep_hidden != 0 (a backward pass will read them); with keep_hidden == 0 their contents are
 * unspecified after the call.  Other shapes use the layered path (one launch per layer), which always needs the
 * h1 / h2 buffers.  ssac_set_fused_forward(0) forces the layered path (cross-check).  Default 1. */
int ssac_set_fused_forward(int on);
int ssac_get_fused_forward(void);
int ssac_mlp_forward(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                     const float* b3, const int32_t* net_index_dev, int G, int D, int H, int O,
                     const float* x_dev, int64_t ldx, int64_t x_gs, int B, float* h1_dev, float* h2_dev,
                     int keep_hidden, float* y_dev, int impl, void* stream);
/* Backward of the above.  dy [G,B,O] (nullable = 0), dh2_extra [G,B,H] (nullable) is added to dL/dh2 scaled
 * by extra_scale (DR3, learning.py:100-108).  Weight grads gW1..gb3 laid out like the parameters (all NULL =
 * input-gradient only, the actor update's pass through the critics); accumulate != 0 adds to them.
 * dx_dev [G,B,D] (nullable) with row stride lddx.  ws_dev: workspace of ssac_mlp_backward_ws(G,B,H) floats. */
int64_t ssac_mlp_backward_ws(int G, int B, int H);
int ssac_mlp_backward(const float* W1, const float* W2, const float* W3, const int32_t* net_index_dev, int G,
                      int D, int H, int O, const float* x_dev, int64_t ldx, int64_t x_gs, int B,
                      const float* h1_dev, const float* h2_dev, const float* dy_dev, const float* dh2_extra_dev,
                      float extra_scale, float* gW1, float* gb1, float* gW2, float* gb2, float* gW3, float* gb3,
                      int accumulate, float* dx_dev, int64_t lddx, float* ws_dev, int impl, void* stream);

/* Split backward of a scalar-output (critic) ensemble, impl 2, D <= 32.  With O == 1 the seed dq[g,b] = dL/dq factors
 * out of the data-gradient chain: dz2 = dq (x) v, dz1 = dq (x) u with v = W3 .* (h2 > 0), u = (v W2) .* (h1 > 0), neither
 * of which depends on the TD target.  _pre computes u into ws_dev (ssac_mlp_backward_ws floats: v then u; v itself is
 * generated from h2 and W3 inside the GEMMs that consume it and only materialised when an operand is not TMA-addressable)
 * and can run next to the target networks; _post needs dq and leaves only the three weight-gradient reductions
 * gW1 = (dq.*u)^T x, gW2 = (dq.*v)^T h1, gW3 = dq^T h2 (+ bias gradients), overwriting the gradient arrays.  Same
 * results as ssac_mlp_backward up to fp32 rounding of dz1 (dq is applied after, not before, the W2 product).
 * u_async != 0 (and ssac_set_overlap on): the u GEMM is forked onto the library's own second stream and joined by the
 * matching _post call (which must follow on a stream ordered after `stream`) -- the output layer, the loss and the gW2
 * reduction do not read u, so it leaves the caller's chain. */
int ssac_mlp_backward_pre(const float* W2, const float* W3, int G, int H, int B, const float* h1_dev, const float* h2_dev,
                          float* ws_dev, int u_async, int impl, void* stream);
int ssac_mlp_backward_post(const float* W3, int G, int D, int H, const float* x_dev, int64_t ldx, int64_t x_gs, int B,
                           const float* h1_dev, const float* h2_dev, const float* dq_dev, float* ws_dev, float* gW1,
                           float* gb1, float* gW2, float* gb2, float* gW3, float* gb3, int impl, void* stream);

/* The actor update's pass through an ensemble of scalar-output critics (learning.py:400-418): from the seed dq [G,B]
 * (ssac_actor_loss_seed: non-zero on each row's arg-min net only) straight to the action gradient summed over the nets,
 * da[b][a] = sum_g dQ_g/dx[b][col0 + a] * dq[g][b], without materialising the per-net input gradients (replaces
 * ssac_mlp_backward(dx only) + ssac_sum_groups).  A <= 32; ws_dev as for ssac_mlp_backward. */
int ssac_mlp_backward_dact(const float* W1, const float* W2, const float* W3, int G, int D, int H, int col0, int A, int B,
                           const float* h1_dev, const float* h2_dev, const float* dq_dev, float* da_dev, float* ws_dev,
                           int impl, void* stream);

/* Actor forward with the policy head fused into the output-layer kernel (one member): replaces ssac_mlp_forward +
 * ssac_tanh_normal_forward / ssac_det_head_forward.  out [B, 2A] (stochastic) or [B, A] (deterministic) is kept for the
 * backward.  deterministic: eps (nullable) is the 1e-4 rsample jitter, noise (nullable) the TD3 noise. */
int ssac_actor_forward_sample(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                              const float* b3, int D, int H, int A, int deterministic, const float* x_dev, int64_t ldx,
                              int B, float* h1_dev, float* h2_dev, int keep_hidden, float* out_dev, const float* eps_dev,
                              const float* noise_dev, float sigma, float clip, float log_std_lo, float log_std_hi,
                              float* a_dev, int64_t lda, float* logp_dev, float* tanh_out_dev, int impl, void* stream);
/* Critic forward of one member (N nets, shared input) with the loss seed of ssac_critic_loss_seed fused into the
 * output-layer kernel: q [N,B], dq [N,B], loss_dev[0] += loss, loss_dev[1] += mean td of the last net.
 * phase 0 = everything; 1 = hidden layers only (h1, h2: independent of the TD target, so the caller can run it on a
 * second stream next to the target networks); 2 = output layer + loss only (h2 from an earlier phase-1 call). */
int ssac_critic_forward_loss(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                             const float* b3, int N, int D, int H, const float* x_dev, int64_t ldx, int B,
                             float* h1_dev, float* h2_dev, float* q_dev, const float* y_dev, const float* w_dev,
                             const float* imp_dev, const float* popart_dev, int pop, int E, int n_total, float* dq_dev,
                             float* loss_dev, int phase, const float* qt_dev, int M, const float* logp_dev,
                             const float* log_alpha_dev, const float* r_dev, const float* d_dev, double gamma,
                             float* y_out_dev, float* td_logs_dev, int impl, void* stream);
/* qt_dev != NULL (phase 2, no PopArt): the TD target of ssac_td_target is evaluated inside the loss kernel instead of
 * being read from y_dev -- y[b] = r[b] + gamma (1 - d[b]) (min_m qt[m][b] - exp(*log_alpha) logp[b]), bit-identical to
 * ssac_td_target -- which takes one dependent launch off the update's critical path.  y_out_dev (nullable) receives y;
 * td_logs_dev[0..2] += {sum_b (y - c), sum_b (y - c)^2, sum_b alpha logp} and td_logs_dev[3] = c = y[0], from which the
 * caller forms the logged mean / unbiased std / entropy bonus (learning_utils.py:351-353). */

/* ---- row-local forwards on the CUDA cores (exact fp32): the single-net, latency-bound pieces ------------------------
 * One launch of ceil(B/16) clusters x 4 CTAs; every cluster walks the whole chain for 16 batch rows (layer slices per CTA,
 * activations exchanged over distributed shared memory).  H in 32..256 (multiple of 8), first-layer width <= 64, O <= 16;
 * ssac_rows_supported(D, H, O) tells.  No activations are kept (forward-only uses).
 * ssac_policy_rows: one actor with its head (acting path agent.py:204-327, forward-only policy samples); out_dev
 * (nullable) receives the raw output layer [B, 2A | A]. */
int ssac_rows_supported(int D, int H, int O);
/* 0: ssac_rows_supported answers 0 for every shape, i.e. callers keep the tensor-core launches (A/B switch).  Default 1. */
int ssac_set_rows_enabled(int on);
int ssac_policy_rows(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3, const float* b3,
                     int D, int H, int A, int deterministic, const float* x_dev, int64_t ldx, int B, float* out_dev,
                     const float* eps_dev, const float* noise_dev, float sigma, float clip, float log_std_lo,
                     float log_std_hi, float* a_dev, int64_t lda, float* logp_dev, float* tanh_out_dev, void* stream);

/* ---- policy heads: nets/distributions.py:9-15,64-114; learning_utils.py:48-59 --------------------- */
/* out [B,2A] = [mu | raw_log_std], eps [B,A] -> a [B,A] (row stride lda: may be a column block of cat(s,a)),
 * logp [B] (sum over A of Normal.log_prob(x) - log|d tanh|).  Saves nothing: backward recomputes. */
int ssac_tanh_normal_forward(const float* out_dev, const float* eps_dev, int B, int A, float log_std_lo,
                             float log_std_hi, float* a_dev, int64_t lda, float* logp_dev, void* stream);
/* d(out) from d(a) [B,A] (row stride ldda, nullable) and d(logp) [B] given as a device scalar multiplier:
 * dlogp[b] = dlogp_scale * exp(*log_alpha_dev) (log_alpha_dev nullable = 1).  rsample path, learning.py:392-399. */
int ssac_tanh_normal_backward(const float* out_dev, const float* eps_dev, int B, int A, float log_std_lo,
                              float log_std_hi, const float* da_dev, int64_t ldda, float dlogp_scale,
                              const float* log_alpha_dev, float* dout_dev, void* stream);
/* log-prob of dataset actions (cache miss: atanh(clamp(a, +-0.99))), AFBC: learning_utils.py:259-267.
 * dlogp_dev nullable: when given also writes d(out) = dlogp * d logp/d out. */
int ssac_tanh_normal_logprob(const float* out_dev, const float* a_dev, int64_t lda, int B, int A, float log_std_lo,
                             float log_std_hi, float* logp_dev, const float* dlogp_dev, float* dout_dev,
                             void* stream);
/* Deterministic actor head (+ optional rsample jitter 1e-4*eps, + optional TD3 noise):
 * a = clamp(tanh(out) [+ 1e-4*eps] + clamp(sigma*noise, +-clip), -1+1e-6, 1-1e-6); clip <= 0 means no clip;
 * noise NULL means no noise / no clamp.  tanh_out_dev (nullable) keeps tanh(out) for the backward. */
int ssac_det_head_forward(const float* out_dev, const float* eps_dev, const float* noise_dev, int B, int A,
                          float sigma, float clip, float* a_dev, int64_t lda, float* tanh_out_dev, void* stream);
/* dout = da * (1 - tanh(out)^2)  (straight-through clamp). */
int ssac_det_head_backward(const float* tanh_out_dev, const float* da_dev, int64_t ldda, int B, int A,
                           float* dout_dev, void* stream);

/* ---- PopArt state: popart.py:8-59.  popart_dev float[4] = {mu, nu, w, b}; popart_ctl_dev int32[2] = {t, stable} */

/* ---- TD target: learning_utils.py:298-354 --------------------------------------------------------- */
/* q_t [M,B] target-critic values on (s1, a1); v = min_M q_t - exp(log_alpha)*logp  (logp NULL: no entropy
 * term, the TD3 branch); PopArt de-normalise if pop; y = r + gamma*(1-d)*v; PopArt update_stats + normalise
 * if popart_dev given.  logs_dev float[3] = {mean(y), std(y) (unbiased), mean(entropy_bonus)}. */
int ssac_td_target(const float* q_t_dev, int M, int B, const float* logp_dev, const float* log_alpha_dev,
                   const float* r_dev, const float* d_dev, float gamma, float* popart_dev, int32_t* popart_ctl_dev,
                   int pop, double popart_beta, int popart_min_steps, float* y_dev, float* logs_dev, void* stream);

/* ---- weighted Bellman backups: learning_utils.py:357-398 ------------------------------------------ */
/* kind 0 'sunrise': q [E,N,B] -> min over N -> unbiased std over E -> sigmoid(-std*T)+0.5
 * kind 1 'softmax': q [E,N,B] -> min over N -> std over E -> B*softmax_batch(-std*T)
 * popart of member j (nullable table popart_dev [E,4]) is NOT applied (the reference does not either).
 * logs_dev float[4] = {mean, max, min, std(unbiased)}. */
int ssac_backup_weights(const float* q_dev, int E, int N, int B, float temperature, int kind, float* w_dev,
                        float* logs_dev, void* stream);

/* ---- critic loss seed: learning.py:90-98,112 ------------------------------------------------------ */
/* q [N,B] predictions of one member, y [B], w [B] (nullable = 1), imp [B] (nullable = 1).
 * q' = popw*q+popb if pop.  dq[k,b] = -2*w*imp*(y-q')*popw * inv_count, inv_count = 1/(B*E*n_total) where n_total
 * is the ensemble-wide number of critics per member (= N unless the critics are sharded over ranks; 0 means N);
 * loss_dev[0] += sum_k mean_b(w*imp*(y-q')^2) * (1/(E*n_total));  loss_dev[1] = mean_b(y - q'_{N-1}). */
int ssac_critic_loss_seed(const float* q_dev, int N, int B, const float* y_dev, const float* w_dev,
                          const float* imp_dev, const float* popart_dev, int pop, int E, int n_total, float* dq_dev,
                          float* loss_dev, void* stream);
/* DR3 feature co-adaptation: f, f1 [N,B,H]: out_dev[0] = mean_{N,B} sum_H f*f1. */
int ssac_dr3_dot(const float* f_dev, const float* f1_dev, int N, int B, int H, float* out_dev, void* stream);

/* ---- actor loss seed: learning.py:400-408 --------------------------------------------------------- */
/* q [N,B] = critics on (s, pi(s)); vals = min_N (popart if pop); dq[k,b] = -(popw)/(E*B) on the arg-min net,
 * 0 elsewhere.  loss_dev[0] += -(1/E) * mean_b(vals - exp(log_alpha)*logp) (logp NULL: no entropy term). */
int ssac_actor_loss_seed(const float* q_dev, int N, int B, const float* logp_dev, const float* log_alpha_dev,
                         const float* popart_dev, int pop, int E, float* vals_dev, float* dq_dev, float* loss_dev,
                         void* stream);
/* out[b, a] = sum_k dx[k, b, col0 + a]   (action-gradient of the arg-min routing, summed over nets). */
int ssac_sum_groups(const float* dx_dev, int G, int B, int64_t lddx, int col0, int A, float* out_dev, void* stream);

/* ---- temperature: learning.py:222-263 ------------------------------------------------------------- */
/* loss = -mean(log_alpha*(logp + target_entropy)); Adam(beta1, beta2) on the scalar, state {m, v} in
 * state_dev float[2], step in ctl_dev int32[2].  logs_dev float[2] = {alpha_loss, exp(new log_alpha)}. */
int ssac_alpha_step(float* log_alpha_dev, const float* logp_dev, int B, float target_entropy, float* state_dev,
                    int32_t* ctl_dev, double lr, double beta1, double beta2, double eps, float* logs_dev, void* stream);

/* ---- advantage filter: adv_estimator.py:58-79, learning_utils.py:241-269,288-295 ------------------ */
/* q_pi [n,B] = min-critic values of n policy samples, q_data [B]: adv = q_data - V with V = mean_n q_pi (method 0,
 * continuous_method "mean") or max_n q_pi (method 1, "max": adv_estimator.py:71-76);
 * mask = (adv >= 0); priority (float64) = relu(adv) + 1e-4.  Any output nullable. */
int ssac_advantage(const float* q_pi_dev, int n, const float* q_data_dev, int B, int method, float* adv_dev,
                   float* mask_dev, double* priority_dev, void* stream);
/* min over the N rows of q [N,B] with optional PopArt affine (agent.py:37-38, adv_estimator.py:30-35). */
int ssac_min_over_nets(const float* q_dev, int N, int B, const float* popart_dev, float* out_dev, void* stream);

/* ---- SAC-Discrete heads: SURVEY 8f N4 (learning_utils.py:322-328, learning.py:84-92, :252-253, :382-390) ---------- */
/* The discrete-action branches run the same grouped MLP launches (ssac_mlp_forward / _backward with O = number of
 * actions A); these entry points are the categorical-policy arithmetic around them.  logits [B,A] row-major = the
 * actor's output (Categorical(logits=...), nets/mlps.py:147-148); actions are stored as floats holding the index
 * (replay row [B,1], read as (int)act[b], clamped to [0,A)).
 *
 * ssac_discrete_value (learning_utils.py:322-328): q_t [M,B,A] target-critic rows of the REDQ subset;
 *   v[b] = sum_a p_a (min_M q_t[.,b,a] - exp(log_alpha) log p_a);  ent_dev[0] += mean_{b,a} exp(log_alpha) log p_a
 *   (nullable; the caller zeroes it).  v then goes through ssac_td_target(M = 1, logp = NULL) for PopArt / r / d. */
int ssac_discrete_value(const float* logits_dev, const float* q_t_dev, int M, int B, int A, const float* log_alpha_dev,
                        float* v_dev, float* ent_dev, void* stream);
/* out[g,b] = q[g,b,act[b]]  (q.gather(-1, a.long()): learning_utils.py:373-376 for the sunrise weights). */
int ssac_discrete_gather_q(const float* q_dev, const float* act_dev, int G, int B, int A, float* out_dev, void* stream);
/* ssac_critic_loss_seed on the gathered Q(s, a_b) (learning.py:90-98): q [N,B,A]; dy [N,B,A] receives the seed at
 * column act[b] and zeros elsewhere (the dense output gradient ssac_mlp_backward takes); loss_dev as there. */
int ssac_discrete_critic_loss_seed(const float* q_dev, int N, int B, int A, const float* act_dev, const float* y_dev,
                                   const float* w_dev, const float* imp_dev, const float* popart_dev, int pop, int E,
                                   int n_total, float* dy_dev, float* loss_dev, void* stream);
/* Actor loss (learning.py:382-390, :408-409): q [N,B,A] online critics on s; vals = popart(min_N q) if pop;
 * f[b] = sum_a p_a (vals_a - exp(log_alpha) log p_a); loss_dev[0] += -(1/E) mean_b f;
 * dlogits[b,k] = -(1/(E B)) p_k ((vals_k - alpha log p_k) - f[b]). */
int ssac_discrete_actor_seed(const float* logits_dev, const float* q_dev, int N, int B, int A, const float* log_alpha_dev,
                             const float* popart_dev, int pop, int E, float* dlogits_dev, float* loss_dev, void* stream);
/* out[b] = sum_a p_a log p_a (learning.py:252-253; feeds ssac_alpha_step as its logp). */
int ssac_discrete_neg_entropy(const float* logits_dev, int B, int A, float* out_dev, void* stream);

/* Indirect advantage of a discrete agent (adv_estimator.py:45-56; filter learning_utils.py:257-262, priorities :288-295):
 * logits [E,B,A] = every actor of the ensemble on the batch, q [N,B,A] = the member's critics; min_q = min_N q with the
 * member's PopArt affine when popart_dev is given; V[b] = sum_a (mean_E p_e[b,a]) min_q[b,a]; adv = min_q[b,act[b]] - V;
 * mask = (adv >= 0); priority (float64) = relu(adv) + 1e-4.  Any output nullable. */
int ssac_discrete_advantage(const float* logits_dev, int E, const float* q_dev, int N, int B, int A, const float* act_dev,
                            const float* popart_dev, float* adv_dev, float* mask_dev, double* priority_dev, void* stream);
/* Filtered behaviour cloning on a categorical policy (learning_utils.py:241-269 with discrete=True):
 * loss_dev[0] += -(1/B) sum_b mask[b] log p[b,act[b]] (mask nullable = 1);
 * dlogits[b,k] = -(mask[b] / (B E)) (1[k = act[b]] - p[b,k]). */
int ssac_discrete_bc_seed(const float* logits_dev, const float* act_dev, const float* mask_dev, int B, int A, int E,
                          float* dlogits_dev, float* loss_dev, void* stream);

/* ---- ensemble sharding over NVLink peer memory: SURVEY 8e (no counterpart in the reference: it is single-device) ---- */
/* The exchanges of the sharded learner (target Q rows, Q(s,pi(s)) rows, dL/da partials, SUNRISE batches / values) as two
 * small kernels over SYMMETRIC buffers (one allocation of 2 x half_bytes per rank, mapped into every peer; the mappings
 * come from torch.distributed._symmetric_memory.rendezvous): no NCCL launch on the update's critical path.
 *   ssac_peer_put : copy nbytes from src_dev to offset dst_off of the current half (epoch parity) of EVERY rank's buffer
 *                   (peer_bufs_dev: device array of `world` mapped pointers, own rank included) with 16-byte peer stores,
 *                   fence at system scope, then raise this rank's signal on every rank: sigs[p][rank] = ++epoch.
 *   ssac_peer_wait: spin until every rank's signal reached the epoch of the preceding put, then copy the first nbytes of
 *                   the current half into out_dev (an address that is stable across CUDA-graph replays) -- or, with
 *                   row_index_dev (device int32[n_rows]), only rows row_index[m] of row_bytes each (the REDQ subset).
 * epoch_dev: device uint32 owned by the exchange site (one per site: sites never share signals).  Both calls are
 * CUDA-graph capturable; ranks run the same sequence of exchanges (lock-step by construction of the sharded update). */
int ssac_peer_put(const void* src_dev, int64_t nbytes, int64_t dst_off, int64_t half_bytes, void* const* peer_bufs_dev,
                  uint32_t* const* peer_sigs_dev, int rank, int world, uint32_t* epoch_dev, void* stream);
int ssac_peer_wait(const void* my_buf_dev, int64_t half_bytes, int64_t nbytes, const uint32_t* my_sigs_dev, int world,
                   const uint32_t* epoch_dev, void* out_dev, const int32_t* row_index_dev, int n_rows, int64_t row_bytes,
                   void* stream);
/* Bulk all-reduce (sum) of n floats for the batch-sharded learner's gradients: dst_dev = sum over the ranks of src_dev
 * (dst may alias src), bitwise identical on every rank.  Two-shot over a symmetric buffer (my_buf_dev on this rank,
 * peer_bufs_dev: device array of the `world` mapped pointers) of 4 x cap_bytes (two epoch halves of {in, out} regions of
 * cap_bytes >= 4n, a multiple of 16): stage src into this rank's `in`; rank r sums its 1/W slice of every rank's `in` in
 * rank order 0..W-1 in fp32 (rank W-1 also the n % 4 tail) and stores it into every rank's `out`; then `out` is copied to
 * dst.  Signals: symmetric uint32[128] per rank (my_sigs_dev / peer_sigs_dev as for put/wait: slots 0..63 "staged",
 * 64..127 "reduced"); epoch_dev as for put/wait; ticket_dev: device uint32[2] of this rank, zero-initialised once (the
 * kernels reset it).  Multi-block, 16-byte loads and stores, no allocation and no host synchronisation (capturable). */
int ssac_peer_allreduce(const float* src_dev, float* dst_dev, int64_t n, void* my_buf_dev, int64_t cap_bytes,
                        void* const* peer_bufs_dev, const uint32_t* my_sigs_dev, uint32_t* const* peer_sigs_dev, int rank,
                        int world, uint32_t* epoch_dev, uint32_t* ticket_dev, void* stream);

/* ---- DrQ pixel encoder: nets/cnns.py:37-69 (BigPixelEncoder), SURVEY 8f N3 ------------------------------------------ */
/* obs [B,C,H,W] fp32 in 0..255 -> obs/255 - 0.5 -> conv3x3 stride 2 (C -> 32) -> 3 x conv3x3 stride 1 (32 -> 32), each + ReLU
 * -> flatten (NCHW order, cnns.py:63) -> Linear(32*h*w, out_dim) -> LayerNorm(eps 1e-5) -> tanh, forward and backward, as
 * implicit GEMMs on the tcgen05 tensor cores (3xTF32, fp32 accumulate) over NHWC activations; replaces the cuDNN / ATen call
 * sequence of BigPixelEncoder.forward and its autograd.  C <= 16, H and W even, out_dim <= 64.
 * params / grads: HOST arrays of 12 device pointers in the module's parameter order: conv1.weight [32,C,3,3], conv1.bias,
 * conv2.weight [32,32,3,3], conv2.bias, conv3.*, conv4.*, fc.weight [out_dim, 32*h*w], fc.bias, ln.weight, ln.bias.
 * ws_dev: caller-owned workspace of ssac_conv_encoder_ws_floats floats, ZERO-INITIALISED once by the caller (padding
 * channels / pixels are never written); it carries the activations from a forward with save = 1 to its backward.
 * save = 0: no backward will follow (target encoder, acting path): activations ping-pong between two buffers.
 * out_dev f32 [B,out_dim].  backward: dout_dev = dL/dout, out_dev = the forward's output, obs_dev = the forward's input (not
 * read: the first layer's weight gradient reads the space-to-depth copy of it that the forward left in ws_dev); every
 * gradient is WRITTEN (not accumulated).  ssac_conv_encoder_ws_offsets (tests / tools): int64[32] = float offsets of {x0, y1..y4, dz1..dz4, wfc,
 * gwfc, fc partials, xhat, rstd, dfc, dl} followed by {rows R1..R4, pitches P1..P4 of the four layers' grids, kf, kf padded,
 * split size, splits, total}.  Layer l works on its INPUT grid R_l x P_l per image: y_l (l = 1..3) is stored compacted on
 * layer l+1's grid, y4 on layer 4's own grid (valid region R4-2 x P4-2), dz_l on layer l's grid. */
/* debugging switch (results do not depend on it): bit 0 = halo tiles (one TMA box per tile instead of one per filter tap) in
 * the forward / data-gradient kernel, bit 1 = in the weight-gradient kernel; a cleared bit forces the per-tap kernel, which
 * otherwise only runs where the halo box does not fit.  mode 0..3, default 3. */
int ssac_set_conv_halo(int mode);
int ssac_conv_encoder_ws_floats(int B, int C, int H, int W, int out_dim, int save, int64_t* n_floats_out);
int ssac_conv_encoder_ws_offsets(int B, int C, int H, int W, int out_dim, int save, int64_t* offsets_out);
int ssac_conv_encoder_forward(const float* obs_dev, int B, int C, int H, int W, int out_dim, const float* const* params,
                              float* ws_dev, int save, float* out_dev, void* stream);
int ssac_conv_encoder_backward(const float* dout_dev, const float* out_dev, const float* obs_dev, int B, int C, int H, int W,
                               int out_dim, const float* const* params, float* ws_dev, float* const* grads, void* stream);

/* ---- host-side helpers of the graph-replayed path (graphed.py) ---------------------------------------------------- */
/* Raw runtime calls behind one C call each (handles: cudaEvent_t / cudaStream_t / cudaGraphExec_t as void*): what a
 * training loop does per update on the host is a graph launch plus a few event operations.
 * ssac_graph_launch: cudaGraphLaunch on `stream` [+ record done_event behind it].
 * ssac_pipelined_launch: record caller_ready_event on caller_stream, make launch_stream wait for it, launch the graph on
 * launch_stream [+ record done_event]: an update that follows everything the caller has issued so far without the
 * caller's stream having to wait for the update (graphed._Cross). */
int ssac_event_record(void* event, void* stream);
int ssac_stream_wait_event(void* stream, void* event);
int ssac_graph_launch(void* graph_exec, void* stream, void* done_event);
int ssac_pipelined_launch(void* graph_exec, void* launch_stream, void* caller_stream, void* caller_ready_event,
                          void* done_event);

#ifdef __cplusplus
}
#endif
#endif /* SSAC_B200_H */
