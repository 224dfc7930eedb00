/*
 * rtk_b200.h - C ABI of the B200 (sm_100a) DPSelect + PivotKV kernels.
 *
 * The reference (SCZwangxiao/video-ReTaKe) is pure Python/PyTorch and has no FFI of its own; every entry
 * point below replaces a span of stock torch ops inside one of its two hot-path operators and is what a
 * ctypes binding in the reference's own modules would call (INTEGRATION.md shows that binding):
 *
 *   retake/visual_compression.py:86-177   memory_bank_compress_keyframe   -> rtk_dpselect_*
 *   retake/visual_compression.py:5-83     memory_bank_compress_MALLM[_hard] (+ the callers' loops) -> rtk_mallm_*
 *   retake/longvideo_cache.py:217-323     PivotKVCache.update             -> rtk_pivot_*
 *
 * Conventions
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers unless the name ends in _host;
 *   - bf16 tensors are passed as `const void*` (2-byte elements), indices are int32, positions int64;
 *   - `stream` is a cudaStream_t passed as void*; every call only enqueues work on it: no allocation, no
 *     host synchronisation, no global state; the caller owns every buffer including `workspace`;
 *   - return value: 0 = ok; >0 = cudaError_t from a launch; <0 = RTK_E_* argument error
 *     (rtk_error_string() turns either into text);
 *   - every compute entry point opens an NVTX range named after itself on the calling thread (visible in nsys / ncu
 *     --nvtx; a no-op without a profiler attached);
 *   - the PivotKV and MA-LLM kernels are launched with programmatic dependent launch (each kernel waits for its
 *     predecessor on the stream with griddepcontrol.wait before touching memory); RTK_NO_PDL=1 in the environment
 *     of the process falls back to plain launches.
 */
#ifndef RTK_B200_H_
#define RTK_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTK_ABI_VERSION 3

#define RTK_E_BADARG      (-1)  /* null pointer / non-positive size                         */
#define RTK_E_ALIGN       (-2)  /* pointer or stride not 16-byte aligned                    */
#define RTK_E_UNSUPPORTED (-3)  /* shape outside the supported envelope (see each function) */
#define RTK_E_WORKSPACE   (-4)  /* workspace too small                                      */
#define RTK_E_DRIVER      (-5)  /* could not obtain cuTensorMapEncodeTiled from the driver  */

int         rtk_version(void);
/* 16 hex digits: SHA-256 over the library's sources (csrc/*.cu, csrc/*.cuh, include/rtk_b200.h; build.py computes it
 * and compiles it in).  bench.py and smoke() print it, and the Python binding refuses a library whose id does not match
 * the sources lying next to it, so a record always says which sources ran. */
const char* rtk_build_id(void);
const char* rtk_error_string(int code);
/* A/B and debugging: pass 2 of the PivotKV scoring skips the key-patch tokens (their score is overwritten with 1.0 before
 * the top-k, longvideo_cache.py:272-274; rtk_pivot_update / _batch with a keymask).  on = 0 / 1 switches that off / on for the
 * process (the RTK_NO_KEY_ELISION=1 environment variable sets the initial state), on < 0 only queries; returns the previous
 * state.  The kept indices are the same either way. */
int         rtk_debug_key_elision(int on);
/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches). */
int64_t     rtk_launch_count(void);

/* ------------------------------------------------------------------------------------------------------
 * DPSelect  (retake/visual_compression.py)
 * ---------------------------------------------------------------------------------------------------- */

/* Adjacent-frame cosine distance; replaces visual_compression.py:98-106
 * (F.cosine_similarity on bf16 + `1 - sim.float()` + the leading row of ones), replaying ATen-CUDA's
 * bf16 rounding chain and fp32 reduction order bit for bit.
 *   x    bf16 [T, N, C] contiguous, 16-byte aligned, C % 8 == 0, 256 <= C <= 8192
 *   halo 0: dis is fp32 [T, N]; row 0 is 1.0, row t is 1 - cos(x[t-1], x[t])
 *        1: x[0] is the last frame owned by the previous rank; dis is fp32 [T-1, N], row j belongs to x[j+1]
 */
int rtk_dpselect_dis(const void* x, int64_t T, int64_t N, int64_t C, int halo, float* dis, void* stream);

/* Peaks + top-t + ascending index list + key-patch mask; replaces visual_compression.py:108-135 (sync=1)
 * and :141-169,175 (sync=0): max_pool1d_with_indices/unique/nonzero, `+= 2`, topk, sort, mask gather.
 *   dis    fp32 [T, N]           (T <= 8192)
 *   t      1 <= t <= T
 *   idx    int32 [t, N] (sync=0) or [t] (sync=1): kept frame index per output slot, ascending in dim 0
 *   mask   uint8 [t * N]: 1 where the kept (frame, patch) is a peak (row-major j * N + p)
 * Peaks replay ATen's max-pool window loop: the window [i-1, i+1] (clipped to [0, T)) starts at its first position with
 * max -inf and takes v when v > max || isnan(v); frame i is a peak when the loop ends on i.  On finite values that is
 * the first maximum; a run of NaNs peaks at the last NaN of each window.
 * Ties at the t-th key are resolved like ATen's CUDA radix select: larger keys first, equal keys by
 * ascending frame index; key order is the radix order (-0 < +0, NaN largest).
 */
int rtk_dpselect_select(const float* dis, int64_t T, int64_t N, int64_t t, int sync,
                        int32_t* idx, uint8_t* mask, void* stream);

/* Stream compaction of the surviving rows; replaces visual_compression.py:138 / :173.
 *   out[j, p, :] = x[idx[j, p], p, :] (sync=0)   or   x[idx[j], p, :] (sync=1);  out bf16 [t, N, C]
 *   t == T (compression_ratio 1.0, the shipped recipe) is the identity; it runs through the same kernel.
 */
int rtk_dpselect_gather(const void* x, int64_t T, int64_t N, int64_t C, const int32_t* idx, int64_t t,
                        int sync, void* out, void* stream);

/* memory_bank_compress_keyframe (visual_compression.py:86-177) as ONE call: rtk_dpselect_dis + _select + _gather launched
 * back to back.  dis (fp32 [T, N]), idx (int32 [t, N] or [t]), mask ([t * N]) and out (bf16 [t, N, C]) are the caller's. */
int rtk_dpselect_keyframe(const void* x, int64_t T, int64_t N, int64_t C, int64_t t, int sync, float* dis,
                          int32_t* idx, uint8_t* mask, void* out, void* stream);

/* Frame-range split of ONE video over the GPUs of a box (SURVEY.md 8e): the compaction of visual_compression.py:138 / :173
 * restricted to the frames a rank owns.  x_local holds frames [frame_first, frame_first + frames_local) of the video (bf16
 * [frames_local, N, C]); idx is the replicated result of rtk_dpselect_select on the all-gathered distances; only the rows of
 * out (bf16 [t, N, C], the reference's layout) whose source frame lies in [t0, t1) are written - the other rows belong to
 * other ranks and are left untouched.  No host synchronisation, no index arithmetic in torch. */
int rtk_dpselect_gather_owned(const void* x_local, int64_t frames_local, int64_t frame_first, int64_t t0, int64_t t1,
                              int64_t N, int64_t C, const int32_t* idx, int64_t t, int sync, void* out, void* stream);

/* Generic row gather out[i, :] = x[src_row[i], :] (rows of row_bytes, a multiple of 16).  Used when DPSelect is split
 * by frame range across GPUs: every rank compacts only the survivors it owns (visual_compression.py:173 restricted
 * to a frame range).  src_row is int64 [rows] on the device. */
int rtk_gather_rows(const void* x, int64_t row_bytes, const int64_t* src_row, int64_t rows, void* out, void* stream);

/* MA-LLM compressors: the caller's loop `while T > t: bank(, size) = memory_bank_compress_MALLM[_hard](...)`
 * (retake/qwen2_vl.py:402-409, retake/llava_onevision.py:235-243 around visual_compression.py:5-47 / :50-83) in one call.
 *   x         bf16 [T, N, C] (not modified);  sizes_in bf16 [T, N] or NULL (= ones): frames each row stands for
 *   t         frames to keep, 1 <= t <= T (t = T - 1 is exactly one call of the reference function)
 *   sync      0: every patch column merges its own most similar adjacent pair;  1: one pair for all patches, chosen on
 *             the bf16 mean of the similarities over the patches (visual_compression.py:21-22)
 *   hard      0: size-weighted average of the pair (:38-46);  1: the first frame of the pair is dropped (:73-79)
 *   out       bf16 [t, N, C];  sizes_out bf16 [t, N] (ignored when hard)
 *   workspace >= rtk_mallm_workspace_bytes(T, N, C, hard) bytes, 256-byte aligned; holds the per-(frame, patch) state
 *             and, for the soft variant, one rewritable copy of the bank.
 * Results are bit-identical to the reference's torch-CUDA op sequence for bf16 banks (every intermediate rounded to
 * bf16, sizes counted in bf16, lowest index among equal similarities). */
size_t rtk_mallm_workspace_bytes(int64_t T, int64_t N, int64_t C, int hard);
int rtk_mallm_compress(const void* x, const void* sizes_in, int64_t T, int64_t N, int64_t C, int64_t t, int sync, int hard,
                       void* out, void* sizes_out, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * PivotKV  (retake/longvideo_cache.py)
 * ---------------------------------------------------------------------------------------------------- */

/* Reverse rotary embedding of a [heads, L, D] bf16 view; replaces longvideo_cache.py:248-259 with
 * apply_(multimodal_)rotary_pos_emb(reverse=True) (:75-77 / :108-110) for ONE of q or k.
 *   x          bf16, element strides (stride_h, stride_l, 1); D even, D % 8 == 0
 *   cos, sin   bf16 [n_pos, L, D] contiguous as returned by rotary_emb (n_pos = 3 mrope, 1 otherwise)
 *   mrope_section int32[3] (host) or NULL; channel block i of sections*2 takes position row i % 3
 *   inv_scale2 = fp32(1 / fp32(attention_scaling ** 2))
 *   forward    0: out = bf16(bf16(bf16(x*cos) - bf16(rot(x)*sin)) * inv_scale2)     (reverse branch)
 *              1: out = bf16(bf16(x*cos) + bf16(rot(x)*sin))                        (forward, :79-81)
 *   out        bf16 [heads, L, D], element strides (out_stride_h, out_stride_l, 1)
 */
int rtk_pivot_rope(const void* x, int64_t heads, int64_t L, int64_t D, int64_t stride_h, int64_t stride_l,
                   const void* cos, const void* sin, int n_pos, const int32_t* mrope_section_host,
                   float inv_scale2, int forward, void* out, int64_t out_stride_h, int64_t out_stride_l,
                   void* stream);

/* Bytes of workspace rtk_pivot_score needs for (H, L). */
size_t rtk_pivot_score_workspace_bytes(int64_t H, int64_t L);

/* Pivot scoring; replaces longvideo_cache.py:260-269: repeat_kv, Q.K^T (tcgen05, bf16 -> fp32 in TMEM),
 * bf16 rounding, / sqrt(D), fp32 softmax over the chunk-local keys (no mask), bf16 rounding, sum over
 * queries, bf16 rounding, mean over the G = H / KVH heads of each KV group, bf16 rounding.
 *   q   bf16 [H, L, D] view, element strides (q_stride_h, q_stride_l, 1), 16-byte aligned, D in {64, 128}
 *   k   bf16 [KVH, L, D] view, element strides (k_stride_h, k_stride_l, 1)
 *   head_scores  bf16 [KVH, L]: line-269 value (per-KV-head scores; the all-gather payload when KV heads
 *                are sharded across GPUs)
 *   1 <= L <= 16384; H % KVH == 0.
 */
int rtk_pivot_score(const void* q, int64_t H, int64_t q_stride_h, int64_t q_stride_l,
                    const void* k, int64_t KVH, int64_t k_stride_h, int64_t k_stride_l,
                    int64_t L, int64_t D, void* head_scores, void* workspace, size_t workspace_bytes,
                    void* stream);

/* Mean over KV heads, key-patch override, top-k, ascending index list; replaces longvideo_cache.py:270-277.
 *   head_scores bf16 [KVH, L] (all KV heads, i.e. after the all-gather when sharded)
 *   keymask     uint8 [L] or NULL (keypatches_mask_chunk); masked scores become 1.0
 *   keep        1 <= keep <= L <= 16384
 *   keep_idx    int32 [keep] ascending;  score_out bf16 [L] or NULL (line-270 value, before the override)
 * Tie rule as in rtk_dpselect_select.
 */
int rtk_pivot_select(const void* head_scores, int64_t KVH, int64_t L, const uint8_t* keymask, int64_t keep,
                     int32_t* keep_idx, void* score_out, void* stream);

/* KV / position compaction; replaces longvideo_cache.py:278-288 and :293-295.
 *   k, v   bf16 [KVH, L, D] views with element strides (stride_h, stride_l, 1), 16-byte aligned rows
 *   k_out, v_out bf16 rows [KVH, keep, D] with element strides (out_stride_h, D, 1): k_out[h, j] = k[h, keep_idx[j]]
 *   pos    int64 [n_pos, L] or NULL;  pos_out int64 [n_pos, keep]
 *   reforge 1: pos_out[0] = m + trunc(fp32(pos_out[0] - m) * fp32(keep / L)), m = min(pos_out[0])
 */
int rtk_pivot_compact(const void* k, const void* v, int64_t KVH, int64_t L, int64_t D,
                      int64_t stride_h, int64_t stride_l, const int32_t* keep_idx, int64_t keep,
                      void* k_out, void* v_out, int64_t out_stride_h,
                      const int64_t* pos, int n_pos, int64_t* pos_out, int reforge, void* stream);

/* Up to four strided bf16 [heads, rows, D] block copies in one launch: the in-place cache append of K and V
 * (DynamicCache.update's torch.cat, longvideo_cache.py:238) and the write of the kept rows over the previous chunk
 * (longvideo_cache.py:313-318).  Arrays have n_jobs entries; strides in elements. */
int rtk_kv_block_copy(int n_jobs, const void* const* src, void* const* dst, const int64_t* heads, const int64_t* rows,
                      const int64_t* src_stride_h, const int64_t* src_stride_l, const int64_t* dst_stride_h,
                      const int64_t* dst_stride_l, int64_t D, void* stream);

/* cos/sin tables of one chunk from the rotary module's inv_freq (fp32 [D/2]); replaces the two
 * `rotary_emb_fn(x, position_ids)` calls of longvideo_cache.py:249,298 plus the mrope row selection of :67-73 when
 * the module is a stock HF rotary embedding with a static inv_freq:
 *   cos_out/sin_out bf16 [L, D]: bf16(cos(fp32(pos[row(c), l]) * inv_freq[c mod D/2]) * attention_scaling)
 */
int rtk_pivot_rope_tables(const int64_t* pos, int n_pos, int64_t L, int64_t D, const float* inv_freq,
                          const int32_t* mrope_section_host, float attention_scaling, void* cos_out, void* sin_out,
                          void* stream);

/* One compressing PivotKVCache.update (longvideo_cache.py:244-306) as a single call: un-rotate, score, select,
 * compact, re-index, re-rotate.  All temporaries live in `workspace` (256-byte aligned). */
typedef struct rtk_pivot_update_args {
    const void* q; int64_t H, q_stride_h, q_stride_l;           /* bf16 [H, L, D] view                              */
    const void* k; int64_t KVH, k_stride_h, k_stride_l;         /* bf16 [KVH, L, D] view                            */
    const void* v; int64_t v_stride_h, v_stride_l;
    int64_t k_stride_h_in, k_stride_l_in;                       /* == k_stride_h/l (kept apart: k is re-pointed)    */
    int64_t L, D;
    const uint8_t* keymask;                                     /* [L] or NULL                                      */
    int64_t keep;
    int32_t reforge;                                            /* pos_embed_reforge                                */
    int32_t n_pos;                                              /* 3 (mrope) or 1; 0 when pos == NULL               */
    const int64_t* pos;                                         /* [n_pos, L] or NULL                               */
    const void* cos; const void* sin;                           /* bf16 [n_pos, L, D] tables, or NULL with inv_freq */
    const float* inv_freq;                                      /* fp32 [D/2] or NULL                               */
    float attention_scaling, inv_scale2;                        /* inv_scale2 = fp32(1 / fp32(scaling ** 2))        */
    int32_t mrope_section[3];
    int32_t skip_select;                                        /* 1: stop after head_scores (KV-head sharding)     */
    void* k_out; void* v_out; int64_t out_stride_h;             /* bf16 [KVH, keep, D]                              */
    int64_t* pos_out;                                           /* [n_pos, keep] or NULL                            */
    int32_t* keep_idx;                                          /* [keep]                                           */
    void* head_scores;                                          /* bf16 [KVH, L]                                    */
    void* workspace; size_t workspace_bytes;
    void* ev_score_begin; void* ev_score_end;                   /* optional cudaEvent_t pair recorded around the scoring   */
    int64_t pos_out_stride;                                     /* row stride of pos_out in elements; 0 = keep (ABI 2)     */
    /* ---- ABI 3: the KV-head split of ONE video over the GPUs of a box (SURVEY.md 8e) as two calls around one exchange.
     * Call 1 (skip_select = 1) scores this rank's KV heads; call 2 (skip_score = 1) selects on the rows of EVERY rank and
     * compacts this rank's heads.  Call 2 must follow call 1 with the same arguments and workspace (the un-rotated K copy of
     * call 1 is compacted).  The exchange in between is either the caller's own collective (xchg_world = 0: e.g. one NCCL
     * all_gather_into_tensor) or done by the library over peer-mapped memory (xchg_world > 1, below).                        */
    int32_t skip_score;                                         /* 1: head_scores is an INPUT, bf16 [score_rows, L]       */
    int32_t score_rows;                                         /* rows averaged by the select (0: KVH)                    */
    /* Peer exchange (NVLink P2P stores, no collective launch): xchg_scores[r] is rank r's bf16 [score_rows, L] buffer and
     * xchg_flags[r] its uint32[8] flag words, both mapped into this process (CUDA IPC / symmetric memory).  Call 1 expects
     * head_scores == (bf16*)xchg_scores[xchg_rank] + xchg_rank * KVH * L, copies those rows into the same rows of every
     * peer's buffer and then stores xchg_epoch into xchg_flags[r][xchg_rank] for every r (release, system scope).  Call 2
     * expects head_scores == xchg_scores[xchg_rank]; its select kernel first waits until all xchg_world words of
     * xchg_flags[xchg_rank] equal xchg_epoch.  Use two buffer / flag sets alternately (a rank may be one update ahead).
     * The wait is bounded: after RTK_XCHG_TIMEOUT_S seconds (environment, default 120, 0 = for ever) the kernel traps and
     * the stream reports a CUDA error - a lost peer must not hang the GPU.                                                 */
    int32_t xchg_world, xchg_rank;
    uint32_t xchg_epoch;
    void* xchg_scores[8];
    uint32_t* xchg_flags[8];
} rtk_pivot_update_args;

/* == rtk_pivot_update_batch_workspace_bytes(H, KVH, L, D, 1) */
size_t rtk_pivot_update_workspace_bytes(int64_t H, int64_t KVH, int64_t L, int64_t D);
/* rtk_pivot_update_batch for one layer: the same launches, workspace layout and argument checks, all of which come before
 * the first launch (a call with skip_select or skip_score is not checked for what only the skipped step reads).  With
 * inv_freq the kept keys come back re-rotated; with cos/sin tables (opaque rotary callable) the caller finishes with
 * rotary_emb_fn(v_out, pos_out) + rtk_pivot_rope(forward=1). */
int rtk_pivot_update(const rtk_pivot_update_args* args, void* stream);

/* The compressing updates of ALL layers of one chunk in one chain of seven launches (deferred compression: the
 * reference's chunk loop calls past_key_values.after_forward() once the chunk's forward is done, retake/qwen2_vl.py:715-716,
 * and a chunk's kept rows are first needed by the NEXT chunk - SURVEY.md 8(f2)).  layers[i] describes layer i exactly as
 * for rtk_pivot_update; H, KVH, L, D, keep, reforge, n_pos, mrope_section and the rotary (inv_freq, attention_scaling)
 * must be the same for every layer, reforge with cos/sin tables instead of inv_freq takes one layer (RTK_E_UNSUPPORTED
 * otherwise: one rtk_pivot_update per layer), pointers
 * and strides are per layer; k_out / v_out may point straight into the layer's cache (rows D apart, heads out_stride_h
 * apart) and pos_out into its position cache (rows pos_out_stride apart).  layers[i].workspace is ignored; `workspace`
 * (256-byte aligned) holds the un-rotated Q / K copies and the row statistics of min(n_layers, 32) layers - more layers
 * run as consecutive groups of 32.  layers[0].ev_score_begin / _end are recorded around the first group's scoring.
 * The KV-head split (ABI 3 fields) works on the whole batch too: skip_select / skip_score / score_rows / xchg_world /
 * xchg_rank / xchg_epoch must agree over the layers, every layer brings its own head_scores rows and xchg_scores buffers,
 * layers[0].xchg_flags carries the one flag set of the call (at most 32 layers then). */
size_t rtk_pivot_update_batch_workspace_bytes(int64_t H, int64_t KVH, int64_t L, int64_t D, int64_t n_layers);
int rtk_pivot_update_batch(const rtk_pivot_update_args* layers, int64_t n_layers, void* workspace, size_t workspace_bytes,
                           void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RTK_B200_H_ */
