/*
 * vfp_b200 - C ABI of the B200 (sm_100a) duplicate-detection hot path.
 *
 * The reference (Alexandre-nk-Perdereau/video-fingerprint) has no FFI layer: its hot path is two Python
 * call sites. Each entry point below replaces the device work behind one of them; the Python host layer in
 * video_fingerprint_b200/ mirrors the reference call signatures and calls these through ctypes
 * (see INTEGRATION.md for the binding a reference maintainer would add).
 *
 *   reference call site                                   replaced by
 *   ----------------------------------------------------  -------------------------------------------
 *   model.load_state_dict(...)      fingerprint.py:70     vfp_weights_create  (BN folding, bf16 packing)
 *   self.model(clip)                fingerprint.py:248    vfp_forward
 *     = VideoFingerprintAttention.forward  model.py:272-298
 *   np.dot(E, E.T) + np.where(>=)   fingerprint.py:493-499  vfp_join_threshold
 *   faiss IndexFlatIP.add/search    fingerprint.py:524-528  vfp_topk_ip
 *
 * Conventions: plain C types only; every buffer is caller-owned; `stream` is a CUDA stream handle
 * (cudaStream_t / CUstream) passed as void*; all device pointers belong to the current device; calls
 * are asynchronous on `stream` and re-entrant (no global mutable state besides the last-error string,
 * which is thread-local). Return value 0 = success, nonzero = error (message via vfp_last_error()).
 * There is no CPU fallback: without a CUDA device every call fails.
 */
#ifndef VFP_B200_H_
#define VFP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VFP_ABI_VERSION 5

/* frame element types accepted by vfp_forward (planar (T,3,64,64) frames as produced by
 * _preprocess_frames, fingerprint.py:186-214; U8 values are scaled by 1/255 on the device) */
#define VFP_FRAME_U8 0
#define VFP_FRAME_BF16 1
#define VFP_FRAME_F32 2
/* decoder layout: (T, 64, 64, 3) uint8, the frames _preprocess_frames holds BEFORE its /255 + permute
 * (fingerprint.py:210-212) - the on-device preprocess of SURVEY.md section 8(f) rank 2 */
#define VFP_FRAME_U8_HWC 3

typedef struct vfp_weights vfp_weights;

/* One entry of the reference checkpoint's model_state_dict (model.py:97-118,129-138,160-175,195-226):
 * `name` is the state_dict key, `data` a HOST pointer to contiguous fp32 values (int64 for
 * num_batches_tracked entries, which are ignored), `numel` the element count. */
typedef struct {
  const char* name;
  const void* data;
  int64_t numel;
} vfp_tensor_desc;

int vfp_abi_version(void);
const char* vfp_last_error(void);

/* Number of SMs of the current device (also a cheap "is there a GPU" probe). Returns <= 0 on failure. */
int vfp_device_sm_count(void);

/* Build the device-resident inference weights from the 144 checkpoint tensors: eval-mode BatchNorm is
 * folded into the preceding conv, Linear(256->S) o Linear(S->256) is folded into one 256x256 map,
 * GEMM operands are packed to bf16 K-major. Blocks until the upload has finished. */
int vfp_weights_create(const vfp_tensor_desc* tensors, int n_tensors, vfp_weights** out);
void vfp_weights_destroy(vfp_weights* w);
/* embedding_dim of the loaded checkpoint (final_projection.3 rows). */
int vfp_weights_embedding_dim(const vfp_weights* w);

/* Device workspace needed to push `frames_per_pass` frames (and up to `clips_per_pass` clips) through
 * the network in one pass. vfp_forward splits its input into passes that fit the workspace it is given;
 * the minimum useful value is the longest clip. About 9 KB per frame plus the frame encoder's scratch for one conv pass
 * (48 KB per frame for min(frames_per_pass, 65 536) frames, + 1 GB that only fp32 frames use); the conv-pass size follows
 * vfp_set_tuning key 3, so size and call under the same setting. */
size_t vfp_forward_workspace_bytes(int64_t frames_per_pass, int64_t clips_per_pass);

/* Fingerprint `n_clips` clips. `frames` is the packed device tensor (sum T, 3, 64, 64) of type
 * `frame_dtype`; `cu_seqlens_host` holds n_clips+1 int32 prefix sums of the clip lengths (HOST memory).
 * Writes unit-norm embeddings (n_clips, D) fp32 to `emb_out` (device). If `features_out` is non-null it
 * receives the temporal features (sum T, 256) fp32 (forward(..., return_features=True), model.py:296-297).
 * Each clip is treated exactly like a B=1 call of the reference module (fingerprint.py:244-249). */
int vfp_forward(const vfp_weights* w, const void* frames, int frame_dtype, const int32_t* cu_seqlens_host,
                int n_clips, float* emb_out, float* features_out, void* workspace, size_t workspace_bytes,
                void* stream);

/* Clips that sit anywhere in device memory, with the conventions of vfp_forward (asynchronous on `stream`, caller-owned
 * buffers, the same pass planner and pipelines): `clip_frames_host` is a HOST array of n_clips device pointers, each at its
 * clip's first frame; frame t of clip i starts `frame_pitch_bytes_host[i]` * t bytes after it (HOST array; NULL = frames back
 * to back). Each frame is one contiguous planar (3, 64, 64) u8 / bf16 / fp32 or decoder-layout (64, 64, 3) u8 frame
 * (VFP_FRAME_U8_HWC). Clips may be separate allocations, windows of one buffer (overlapping or repeated) or views with a
 * frame stride such as every 3rd frame; no frame is copied. Row i of `emb_out` (and rows sum_{j<i} T_j .. of
 * `features_out`, if non-null) have the bits vfp_forward gives for the same frames packed. Size the workspace with
 * vfp_forward_workspace_bytes. A null or not 16-byte aligned pointer, a pitch below one frame or not a multiple of 16, a
 * length below 1 or above the positional table, a workspace too small for the longest clip and an unknown frame_dtype are
 * errors naming the clip, reported before anything is enqueued; beyond that the pointers are not validated (each must
 * address lengths_host[i] readable frames on the current device). */
int vfp_forward_clips(const vfp_weights* w, const void* const* clip_frames_host, const int64_t* frame_pitch_bytes_host,
                      const int32_t* lengths_host, int n_clips, int frame_dtype, float* emb_out, float* features_out,
                      void* workspace, size_t workspace_bytes, void* stream);

/* All-pairs cosine/inner-product threshold join of a query row block against a database:
 * emits every (i, j, s) with s = <q_i, db_j> >= thr computed in fp32, i = q_row0 + local row (so a
 * row-block shard reports global indices). `q`/`db` are device fp32 (n, dim) row-major, dim == 256.
 * `screen_margin` must be >= 2^-8 * max|q_i| * max|db_j| (0.004 for unit vectors): the tensor-core
 * screen runs in bf16 at thr - screen_margin and survivors are re-scored in fp32.
 * counts_out (device, 2 x uint64): [0] = number of result pairs (may exceed `capacity`; only the first
 * `capacity` are stored, in no particular order), [1] = number of screen candidates (if it exceeds the
 * candidate capacity implied by the workspace the result is incomplete and the caller must retry with
 * the workspace vfp_join_workspace_bytes(..., candidates) reports). */
size_t vfp_join_workspace_bytes(int64_t n_q, int64_t n_db, int64_t candidate_capacity);
int vfp_join_threshold(const float* q, const float* db, int64_t n_q, int64_t n_db, int dim, int64_t q_row0,
                       float thr, float screen_margin, int32_t* out_i, int32_t* out_j, float* out_s,
                       int64_t capacity, uint64_t* counts_out, void* workspace, size_t workspace_bytes,
                       void* stream);

/* Exact flat inner-product top-k (the arithmetic of faiss.IndexFlatIP.search): for every query row the k
 * largest <q_i, db_j> in fp32, sorted by (score descending, index ascending). out_s (n_q, k) fp32,
 * out_idx (n_q, k) int64, device memory. k <= 32, dim == 256. The tensor-core screen keeps the 64 best bf16 scores
 * per query, which are re-scored in fp32; `flags_out` (device, 2 x uint64): [0] = query rows whose exactness could
 * not be proven from the screen bound (`screen_margin`, as for the join) and were recomputed by the exact fp32
 * scan, [1] != 0 = that fallback overflowed (more than 8192 such rows or more than 512 tied candidates for one
 * row) and the result must be discarded. */
size_t vfp_topk_workspace_bytes(int64_t n_q, int64_t n_db, int k);
int vfp_topk_ip(const float* q, const float* db, int64_t n_q, int64_t n_db, int dim, int k,
                float screen_margin, float* out_s, int64_t* out_idx, uint64_t* flags_out, void* workspace,
                size_t workspace_bytes, void* stream);

/* VideoFingerprint3D, the reference's second model behind create_model("3d" | "cnn3d") (/root/reference/model.py:406-512):
 * Conv3d(3->16, (fs,5,5), stride (fs,2,2)) / (16->32) / (32->64, temporal stride 2) / (64->128), each + BatchNorm3d(eval) +
 * ReLU, spatial average pool, temporal Conv1d(128,128,3), attention + average pooling over time, Linear-ReLU-Linear
 * projector, L2 normalisation. vfp3d_weights_create takes the model's named fp32 state_dict tensors (like
 * vfp_weights_create) and its frame_stride; vfp3d_forward fingerprints n_clips clips of n_frames frames each
 * (`frames`: device (n_clips*n_frames, 3, 64, 64) planar u8 / bf16 / fp32; T is zero-padded to a multiple of frame_stride
 * like model.py:468-471) into `emb_out` (n_clips, D) fp32, walking the batch in as many passes as the workspace allows. */
typedef struct vfp3d_weights vfp3d_weights;
int vfp3d_weights_create(const vfp_tensor_desc* tensors, int n_tensors, int frame_stride, vfp3d_weights** out);
void vfp3d_weights_destroy(vfp3d_weights* w);
int vfp3d_weights_embedding_dim(const vfp3d_weights* w);
size_t vfp3d_forward_workspace_bytes(const vfp3d_weights* w, int64_t clips_per_pass, int n_frames);
int vfp3d_forward(const vfp3d_weights* w, const void* frames, int frame_dtype, int64_t n_clips, int n_frames,
                  float* emb_out, void* workspace, size_t workspace_bytes, void* stream);

/* Variable-length batches of the 3-D model, with the conventions of vfp_forward: `frames` is the packed device tensor
 * (sum T, 3, 64, 64) planar u8 / bf16 / fp32 (VFP_FRAME_U8_HWC is rejected), clips back to back; `cu_seqlens_host` holds
 * n_clips+1 int32 prefix sums of the clip lengths (HOST memory, cu_seqlens_host[0] = 0). Writes unit-norm embeddings
 * (n_clips, D) fp32 to `emb_out`. Every clip is treated exactly like a B=1 vfp3d_forward on that clip alone, with the same
 * bits: its zero padding up to a multiple of frame_stride and its temporal padding stop at its own ends, whatever surrounds
 * it. A clip may have 1 .. 64 * frame_stride frames (at most 32 temporal positions after the strides); a clip of length 0,
 * a longer clip, decreasing prefix sums, or a workspace too small for a clip are errors naming the clip. `frames` must be
 * 16-byte aligned (the frames are read in 8- and 16-byte vectors); so must vfp3d_forward's. Every torch allocation and
 * every whole-frame view of one is.
 * The call splits the input into passes on clip boundaries that fit `workspace_bytes`; results do not depend on the split.
 * vfp3d_forward_packed_workspace_bytes bounds one pass of up to `frames_per_pass` frames in up to `clips_per_pass` clips
 * (from sum ceil(T/fs) <= F/fs + C and sum T3 <= (sum G + C)/2); the minimum useful value is that of the longest clip
 * (frames_per_pass = its length, clips_per_pass = 1). vfp3d_forward is this path with uniform lengths. */
size_t vfp3d_forward_packed_workspace_bytes(const vfp3d_weights* w, int64_t frames_per_pass, int64_t clips_per_pass);
int vfp3d_forward_packed(const vfp3d_weights* w, const void* frames, int frame_dtype, const int32_t* cu_seqlens_host,
                         int n_clips, float* emb_out, void* workspace, size_t workspace_bytes, void* stream);

/* Clips that sit anywhere in device memory, with the conventions of vfp3d_forward_packed: `clip_frames_host` is a HOST
 * array of n_clips device pointers, each at its clip's first frame, and clip i is `lengths_host[i]` contiguous frames from
 * there, planar (T, 3, 64, 64) u8 / bf16 / fp32 or decoder-layout (T, 64, 64, 3) u8 (VFP_FRAME_U8_HWC, the output of
 * vfp_preprocess_frames; it gives the same bits as the same frames permuted to planar u8). Clips may be separate
 * allocations, overlapping windows of one buffer, or the same frames listed twice; no frame is copied. Row i of `emb_out`
 * has the bits of a B=1 vfp3d_forward on clip i alone. Size the workspace with vfp3d_forward_packed_workspace_bytes
 * (frames_per_pass = the sum of the lengths of a pass). A null or not 16-byte aligned pointer, a length below 1 or above
 * 64 * frame_stride, a workspace too small for a clip and an unknown frame_dtype are errors naming the clip; beyond that
 * the pointers are not validated (each must address lengths_host[i] readable frames on the current device). */
int vfp3d_forward_clips(const vfp3d_weights* w, const void* const* clip_frames_host, const int32_t* lengths_host,
                        int n_clips, int frame_dtype, float* emb_out, void* workspace, size_t workspace_bytes, void* stream);

/* Frame preprocessing of the scanner (/root/reference/fingerprint.py:186-214 _preprocess_frames): cv2.resize(frame,
 * INTER_AREA) so that the short side becomes 64 (new size truncated with int() like the reference), then the centre
 * 64 x 64 crop. `frames_hwc`: device uint8 (n_frames, height, width, 3), all frames of one size; `out_hwc64`: device
 * uint8 (n_frames, 64, 64, 3), which vfp_forward, vfp_forward_clips and vfp3d_forward_clips accept as VFP_FRAME_U8_HWC (the /255 and the
 * HWC->CHW permute of fingerprint.py:210-212 happen inside the first layer's loader). Bit-exact with OpenCV 4.x INTER_AREA: down-scaling (general,
 * integer-factor and 2 x 2 code paths) and, for frames with a side below 64 pixels, the up-scaling branch (8-bit fixed-point
 * bilinear kernels with the area coefficient rule). */
size_t vfp_preprocess_workspace_bytes(int height, int width);
int vfp_preprocess_frames(const uint8_t* frames_hwc, int n_frames, int height, int width, uint8_t* out_hwc64,
                          void* workspace, size_t workspace_bytes, void* stream);

/* Evaluation metrics over an embedding set - the trainer's use of the same N x N similarity matrix
 * (/root/reference/train.py:285-358 compute_discrimination_metrics, :439-481 _compute_retrieval_metrics), computed
 * without storing the matrix. All scores are exact fp32 (one fmaf chain over k = 0 .. dim-1).
 * vfp_pair_scores: out_s[t] = <e[pair_i[t]], e[pair_j[t]]> for m listed pairs (device arrays).
 * vfp_pair_stats: one pass over every ordered pair (i, j), i != j. A "positive" of row i is a column with the same
 * video id; the caller lists them in CSR form (row_ptr (n+1), pos_idx (m), device) with their scores pos_score (m)
 * from vfp_pair_scores and the same scores sorted ascending (sorted_intra (m)). Outputs (device):
 *   rank_greater[q]    = #{j != i : s_ij >  pos_score[q]}             (-> rank of the positive, R@k, mAP)
 *   rank_tie_before[q] = #{j != i, j < pos_idx[q] : s_ij == pos_score[q]}
 *   sums[4]   = sum / sum of squares of the intra-video scores, then of the inter-video scores (double)
 *   counts[20] = n_intra, n_inter, sum over inter scores s of #{intra <= s}, of #{intra < s} (-> AUC-ROC in its
 *                Mann-Whitney form), then for each of the <= 8 thresholds #{intra >= thr} (8 slots) and #{inter >= thr}.
 * `thresholds` is a HOST array of n_thresholds floats. dim must be a multiple of 16, e 16-byte aligned. */
int vfp_pair_scores(const float* e, int64_t n, int dim, const int32_t* pair_i, const int32_t* pair_j, int64_t m,
                    float* out_s, void* stream);
int vfp_pair_stats(const float* e, const int32_t* video_ids, int64_t n, int dim, const int32_t* row_ptr,
                   const int32_t* pos_idx, const float* pos_score, const float* sorted_intra, int64_t m,
                   const float* thresholds, int n_thresholds, uint32_t* rank_greater, uint32_t* rank_tie_before,
                   double* sums, uint64_t* counts, void* stream);

/* Stage profiler (measurement hook, used by bench.py): when enabled, vfp_forward records CUDA events between
 * its stages on the caller's stream. vfp_profile_read synchronises on the last event and returns the accumulated
 * milliseconds per stage (vfp_profile_num_stages entries, names via vfp_profile_stage_name) and the number of
 * kernels vfp_forward / vfp_join_threshold / vfp_topk_ip have launched since the last reset. Not thread-safe. */
int vfp_profile_enable(int on);
int vfp_profile_num_stages(void);
const char* vfp_profile_stage_name(int i);
int vfp_profile_read(double* stage_ms, int n_stages, uint64_t* launches, int reset);

/* Tuning knobs for experiments (process-wide; defaults in parentheses). key 0: frames per conv1+conv2 pass of the two-kernel
 * stem (16384, >= 64); key 1: conv1+conv2 stem: 2 = fused kernel, conv1 as TS-mode tcgen05 UMMA (default for u8 / bf16 frames),
 * 0 = two kernels (always used for fp32 frames); key 2: 1 = hang diagnosis mode (see vfp_debug_hang_log), 0 = watchdog traps
 * (default); key 3: frames per conv pass (64..262144, default 65536); key 5 / key 6: L2 prefetch distance in column tiles of the
 * one-CTA join kernel / the top-k screen for databases larger than L2 (0 = off); key 7: programmatic dependent launch between
 * the forward's kernels (0); key 8: cap on the CTAs of persistent kernels (0 = one per SM); key 9: conv passes in flight on
 * separate streams (1); key 10: join kernel, 0 = one CTA per tile, 1 = A-resident, 2 = A-resident CTA pairs (2); key 11:
 * self joins compute the upper triangle and mirror the pairs (1); key 12: join panel width in column tiles (512); key 13:
 * TMA multicast of the conv3 / conv4 filter tile across a CTA pair, bit mask (0); key 14: 1 = both MLP linears in one kernel (1);
 * key 15: CTA-pair GEMM, bit 0 conv4, bit 1 QKV / out-projection (1); key 16: conv3 with its filters in tensor memory (1);
 * key 17: attention on tcgen05 (1) or the mma.sync twin kept for cross-checks (0).
 * Every setting produces the same results up to fp32 summation order (scripts/dev_tuning_parity.py). */
int vfp_set_tuning(int key, long long value);

/* Reads and clears the device-side error word set by a kernel watchdog (0 = none). Synchronises. */
unsigned int vfp_device_error_word(void);

/* Hang diagnosis (development aid). After vfp_set_tuning(2, 1) a kernel whose mbarrier wait times out logs
 * (barrier shared-memory address, parity, threadIdx.x, blockIdx.x) and abandons the wait instead of trapping;
 * this returns up to max_entries such 4-word records (at most 64 are kept), or -1 on a CUDA error. Synchronises. */
int vfp_debug_hang_log(unsigned int* out, int max_entries);

#ifdef __cplusplus
}
#endif
#endif /* VFP_B200_H_ */
