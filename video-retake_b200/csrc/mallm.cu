// MA-LLM memory-bank compressors (sm_100a): the `compression_method: MA-LLM / MA-LLM-hard` branch of
// compress_video_tokens (retake/qwen2_vl.py:402-409, retake/llava_onevision.py:235-243), i.e. the loop
//     while T > tgt: bank, size = memory_bank_compress_MALLM(bank, size, sync)      (visual_compression.py:5-47)
//     while T > tgt: bank = memory_bank_compress_MALLM_hard(bank, sync)             (visual_compression.py:50-83)
// fused into one call.  The reference recomputes every cosine similarity and rewrites the whole bank on every
// round (O(rounds * T*N*C) bytes); here the bank is read once and each round only touches what changed:
//
//   * state per (frame i, patch p): similarity to the next surviving frame, norm, size, next/prev links, flags;
//   * a round = argmax over the similarities (lowest index among equals, NaN first - torch.max on CUDA), the merge
//     of frames m and next(m), and the replay of the reference's `x = rd(rd(x * size) / size)` on the rows for
//     which that map is not yet at a fixed point (it is idempotent after one or two applications, so the "dirty"
//     list holds the rows changed in the previous round only), then the similarities next to changed rows;
//   * one round body (mallm_round) serves both modes, over a patch column whose state lives in shared memory or in
//     the workspace: patch-local mode runs all rounds of a patch column inside one CTA of one launch, the state in
//     shared memory; sync mode shares one argmax over the bf16 mean of the similarities across patches (one argmax
//     kernel + one round kernel per round, the state in the workspace).
//
// Arithmetic is the reference's, bit for bit (bf16 bank): rd() = round to nearest even to bf16 after EVERY op,
// true fp32 division, sizes kept in bf16; cosine similarity as in dpselect.cu (ATen reduction orders: 4-element
// vectors for the norm, 8-element vectors for the product sum); the sync mean replays ATen's bf16 mean(-1)
// (8-element vectors, block width min(last_pow2(N/8), 32), unaligned head / tail by the row's position in the
// CURRENT bank - which is why all means are refreshed every round when N % 8 != 0).
#include <math.h>

#include "rtk_common.cuh"

namespace rtk {

constexpr int kMlWarps = 8;
constexpr int kMlThreads = kMlWarps * kWarp;

struct MallmParams {
    const __nv_bfloat16* x;          // [T, N, C] input bank (never written)
    __nv_bfloat16* work;             // [T, N, C] rows rewritten by merges (soft mode only)
    const __nv_bfloat16* sizes_in;   // [T, N] or null (= ones)
    int T, N, C;
    long long si, sp;                // strides of the per-(frame, patch) state arrays
    float* sim;                      // similarity to the next surviving frame, -inf when there is none
    float* nrm;                      // clamped bf16 norm of the current row
    float* size;                     // bf16-valued
    int* next;                       // T = none
    int* prev;                       // -1 = none
    uint8_t* alive;
    uint8_t* in_work;
    int* dirty;                      // [2][N][T] rows changed in the previous round
    int* n_dirty;                    // [2][N]
    int* merge_at;                   // sync mode: the shared argmax
    float* msim;                     // [T] sync mode: bf16 mean over patches
    int* touched;                    // [T] sync mode: stamp of the last round that rewrote sim[i][*]
    int sync, hard;
};

__device__ __forceinline__ size_t at(const MallmParams& P, int i, int p) { return (size_t)i * P.si + (size_t)p * P.sp; }

// clamp_min_(bf16(1e-8)) of F.cosine_similarity
__device__ __forceinline__ float clamp_norm(float ss) {
    return fmaxf(round_bf16(__fsqrt_rn(ss)), __uint_as_float(0x322c0000u));
}
__device__ __forceinline__ float warp_tree(float v, int lane) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    return __shfl_sync(0xffffffffu, v, 0);
}

// Rows live in HBM / L2 and every loop below is a chain of dependent round trips unless the loads are issued in
// batches: kBatch independent vector loads per lane are in flight before the first one is consumed.  The order in
// which values enter the accumulators is unchanged (ascending vector index per lane).
constexpr int kBatch = 14;

// norm of one row, ATen order with 4-element vectors (lane l owns the 8-byte vectors l, l+32, ...)
__device__ __forceinline__ float warp_row_norm(const __nv_bfloat16* row, int C, int lane) {
    const uint2* r = reinterpret_cast<const uint2*>(row);
    const int nv = C >> 2;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int v = lane;
    for (; v + (kBatch - 1) * 32 < nv; v += kBatch * 32) {
        uint2 q[kBatch];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) q[u] = r[v + 32 * u];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) {
            fma_sq_bf16x2(a0, a1, q[u].x);
            fma_sq_bf16x2(a2, a3, q[u].y);
        }
    }
    for (; v < nv; v += 32) {
        const uint2 q = r[v];
        fma_sq_bf16x2(a0, a1, q.x);
        fma_sq_bf16x2(a2, a3, q.y);
    }
    return clamp_norm(warp_tree(((a0 + a1) + a2) + a3, lane));
}

// bf16 cosine similarity of two rows given their clamped norms, ATen order with 8-element vectors
__device__ __forceinline__ float warp_pair_sim(const __nv_bfloat16* ra, float na, const __nv_bfloat16* rb, float nb, int C,
                                               int lane) {
    const uint4* A = reinterpret_cast<const uint4*>(ra);
    const uint4* B = reinterpret_cast<const uint4*>(rb);
    const int nv = C >> 3;
    const float ia = __frcp_rn(na), ib = __frcp_rn(nb);      // x * rcp(n) == x / n after the bf16 rounding (DESIGN.md)
    float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f, c4 = 0.f, c5 = 0.f, c6 = 0.f, c7 = 0.f;
    auto step = [&](const uint4& a, const uint4& b) {
        add_bf16x2(c0, c1, mul_bf16x2_rn(scale_bf16x2_rn(a.x, ia), scale_bf16x2_rn(b.x, ib)));
        add_bf16x2(c2, c3, mul_bf16x2_rn(scale_bf16x2_rn(a.y, ia), scale_bf16x2_rn(b.y, ib)));
        add_bf16x2(c4, c5, mul_bf16x2_rn(scale_bf16x2_rn(a.z, ia), scale_bf16x2_rn(b.z, ib)));
        add_bf16x2(c6, c7, mul_bf16x2_rn(scale_bf16x2_rn(a.w, ia), scale_bf16x2_rn(b.w, ib)));
    };
    constexpr int kHalf = kBatch / 2;
    int v = lane;
    for (; v + (kHalf - 1) * 32 < nv; v += kHalf * 32) {
        uint4 a[kHalf], b[kHalf];
#pragma unroll
        for (int u = 0; u < kHalf; ++u) { a[u] = A[v + 32 * u]; b[u] = B[v + 32 * u]; }
#pragma unroll
        for (int u = 0; u < kHalf; ++u) step(a[u], b[u]);
    }
    for (; v < nv; v += 32) step(A[v], B[v]);
    return round_bf16(warp_tree(((((((c0 + c1) + c2) + c3) + c4) + c5) + c6) + c7, lane));
}

// ---------------------------------------------------------------------------------------------- argmax
struct Best {
    float v;
    int i;
};
// torch.max(dim) on CUDA: NaN is the maximum, equal values go to the lowest index
__device__ __forceinline__ bool better(const Best& a, const Best& b) {
    const bool an = a.v != a.v, bn = b.v != b.v;
    if (an || bn) return (an && bn) ? a.i < b.i : an;
    return (a.v != b.v) ? a.v > b.v : a.i < b.i;
}
// argmax over v[i * stride], i < T; the result is valid in every thread.  `scratch` holds one Best per warp.
__device__ __forceinline__ int block_argmax(const float* v, long long stride, int T, Best* scratch) {
    Best b{-INFINITY, 0x7fffffff};
    for (int i = threadIdx.x; i < T; i += blockDim.x) {
        const Best c{v[(size_t)i * stride], i};
        if (better(c, b)) b = c;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        Best o{__shfl_down_sync(0xffffffffu, b.v, off), __shfl_down_sync(0xffffffffu, b.i, off)};
        if (better(o, b)) b = o;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    if (lane == 0) scratch[warp] = b;
    __syncthreads();
    if (warp == 0) {
        b = (lane < nw) ? scratch[lane] : Best{-INFINITY, 0x7fffffff};
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            Best o{__shfl_down_sync(0xffffffffu, b.v, off), __shfl_down_sync(0xffffffffu, b.i, off)};
            if (better(o, b)) b = o;
        }
        if (lane == 0) scratch[0] = b;
    }
    __syncthreads();
    const int r = scratch[0].i;
    __syncthreads();
    return r;
}

// ------------------------------------------------------------------------------------------------ init
// links, sizes, flags, dirty lists (norms and similarities come from the streaming cosine kernel of dpselect.cu,
// which reads the bank once at HBM speed)
__global__ void __launch_bounds__(kMlThreads) mallm_init_kernel(MallmParams P) {
    pdl_enter();
    __shared__ int s_cnt;
    const int p = blockIdx.x;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < P.T; i += blockDim.x) {
        const size_t a = at(P, i, p);
        P.next[a] = i + 1;
        P.prev[a] = i - 1;
        P.alive[a] = 1;
        if (i == P.T - 1) P.sim[a] = -INFINITY;
        if (!P.hard) {
            const float s = P.sizes_in ? __bfloat162float(P.sizes_in[(size_t)i * P.N + p]) : 1.0f;
            P.size[a] = s;
            P.in_work[a] = 0;
            if (s != 1.0f) P.dirty[(size_t)p * P.T + atomicAdd(&s_cnt, 1)] = i;       // not known to be a fixed point
        }
        if (P.sync && p == 0) P.touched[i] = 0;
    }
    __syncthreads();
    if (threadIdx.x == 0 && !P.hard) P.n_dirty[p] = s_cnt;
}

// ----------------------------------------------------------------------------------------------- round
__device__ __forceinline__ uint32_t merge_pair(uint32_t a, uint32_t b, float sa, float sb, float snew) {
    const float lo = round_bf16(__fdiv_rn(round_bf16(round_bf16(bf16lo_to_f32(a) * sa) + round_bf16(bf16lo_to_f32(b) * sb)), snew));
    const float hi = round_bf16(__fdiv_rn(round_bf16(round_bf16(bf16hi_to_f32(a) * sa) + round_bf16(bf16hi_to_f32(b) * sb)), snew));
    return pack_bf16x2_rn(lo, hi);
}
__device__ __forceinline__ uint32_t rescale_pair(uint32_t a, float s) {
    const float lo = __fdiv_rn(round_bf16(bf16lo_to_f32(a) * s), s);
    const float hi = __fdiv_rn(round_bf16(bf16hi_to_f32(a) * s), s);
    return pack_bf16x2_rn(lo, hi);
}

// Row i of patch p: the input row, or its copy in the workspace once a merge or replay has rewritten it.
__device__ __forceinline__ const __nv_bfloat16* bank_row(const MallmParams& P, int i, int p, bool in_work) {
    const size_t off = ((size_t)i * P.N + p) * (size_t)P.C;
    return in_work ? P.work + off : P.x + off;
}
__device__ __forceinline__ __nv_bfloat16* work_row(const MallmParams& P, int i, int p) {
    return P.work + ((size_t)i * P.N + p) * (size_t)P.C;
}

// The state of one patch column, as the round body sees it.  Two implementations: GlobalColumn reads and writes the
// workspace arrays (sync mode, where every round is its own launch), SmemColumn keeps the column in shared memory for
// all rounds of one launch (patch-local mode) and mirrors to the workspace only what mallm_emit_kernel reads.
struct GlobalColumn {
    const MallmParams& P;
    const int p;
    __device__ GlobalColumn(const MallmParams& P_, int p_) : P(P_), p(p_) {}
    __device__ float& sim(int i) const { return P.sim[at(P, i, p)]; }
    __device__ float& nrm(int i) const { return P.nrm[at(P, i, p)]; }
    __device__ int& next(int i) const { return P.next[at(P, i, p)]; }
    __device__ int& prev(int i) const { return P.prev[at(P, i, p)]; }
    __device__ float size(int i) const { return P.size[at(P, i, p)]; }
    __device__ void set_size(int i, float s) const { P.size[at(P, i, p)] = s; }
    __device__ const __nv_bfloat16* row(int i) const { return bank_row(P, i, p, !P.hard && P.in_work[at(P, i, p)]); }
    __device__ void set_in_work(int i) const { P.in_work[at(P, i, p)] = 1; }
    // the rows whose similarity changed in round r: mallm_sync_argmax_kernel refreshes their mean
    __device__ void stamp(int i, int r) const { P.touched[i] = r + 1; }
    __device__ void kill(int i, int r) const {
        P.alive[at(P, i, p)] = 0;
        sim(i) = -INFINITY;
        stamp(i, r);
    }
    // dirty lists [2][N][T] with their counts [2][N]: list r & 1 is read in round r, list (r + 1) & 1 written
    __device__ int n_dirty(int r) const { return P.n_dirty[(size_t)(r & 1) * P.N + p]; }
    __device__ int dirty(int r, int k) const { return P.dirty[((size_t)(r & 1) * P.N + p) * P.T + k]; }
    __device__ void set_dirty(int r, int k, int i) const { P.dirty[((size_t)(r & 1) * P.N + p) * P.T + k] = i; }
    __device__ void end_round(int r, int nch) const {
        if (threadIdx.x == 0) P.n_dirty[(size_t)((r + 1) & 1) * P.N + p] = nch;
    }
};

struct SmemColumn {
    const MallmParams& P;
    const int p;
    float *sim_, *nrm_, *size_;
    int *next_, *prev_;
    short* dirty_;               // [2][T]
    uint8_t* in_work_;
    int nd;                      // length of the dirty list the next round reads
    __device__ float& sim(int i) const { return sim_[i]; }
    __device__ float& nrm(int i) const { return nrm_[i]; }
    __device__ int& next(int i) const { return next_[i]; }
    __device__ int& prev(int i) const { return prev_[i]; }
    __device__ float size(int i) const { return size_[i]; }
    __device__ void set_size(int i, float s) const {
        size_[i] = s;
        P.size[at(P, i, p)] = s;
    }
    __device__ const __nv_bfloat16* row(int i) const { return bank_row(P, i, p, !P.hard && in_work_[i]); }
    __device__ void set_in_work(int i) const {
        in_work_[i] = 1;
        P.in_work[at(P, i, p)] = 1;
    }
    __device__ void stamp(int, int) const {}
    __device__ void kill(int i, int) const {
        P.alive[at(P, i, p)] = 0;
        sim_[i] = -INFINITY;
    }
    __device__ int n_dirty(int) const { return nd; }
    __device__ int dirty(int r, int k) const { return dirty_[(size_t)(r & 1) * P.T + k]; }
    __device__ void set_dirty(int r, int k, int i) const { dirty_[(size_t)(r & 1) * P.T + k] = (short)i; }
    __device__ void end_round(int, int nch) { nd = nch; }
};

// Shared memory of patch-local mode: the column state (25 bytes per frame), then kBufs row buffers.  The host sizes the
// launch with `bytes`, the kernel carves its arrays at the offsets.
struct RoundsSmem {
    size_t sim, nrm, size, next, prev, dirty, in_work, rowbuf, bytes;
};
__host__ __device__ inline RoundsSmem rounds_smem(int T, int C, int bufs) {
    const size_t t4 = (size_t)T * 4;
    RoundsSmem L;
    L.sim = 0;
    L.nrm = t4;
    L.size = 2 * t4;
    L.next = 3 * t4;
    L.prev = 4 * t4;
    L.dirty = 5 * t4;
    L.in_work = 6 * t4;
    L.rowbuf = ((size_t)T * 25 + 15) & ~(size_t)15;
    L.bytes = (size_t)T * 25 + 16 + (size_t)bufs * C * 2 + 16;
    return L;
}

// One round on one patch column, by the whole CTA; m is the frame the round merges (soft) or drops (hard).
// Soft: the merge of (m, next(m)) into m and the replay of x = rd(rd(x * s) / s) on the dirty rows are element-wise over
// the whole CTA, kBufs rows per batch with every load of the batch in flight at once; each result goes to the workspace
// row AND to a shared row buffer (`rowbuf`, kBufs * C bf16) from which one warp per row takes the norm in ATen's order.
// Then the similarities on both sides of every changed row, one warp per pair.  Hard: one pair similarity.
template <int kBufs, class Col>
__device__ __forceinline__ void mallm_round(const MallmParams& P, Col& c, __nv_bfloat16* rowbuf, int r, int m) {
    __shared__ int s_cnt, s_changed[kBufs];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int T = P.T, C = P.C, nv = C >> 2;
    if (P.hard) {
        if (warp == 0) {
            const int pm = c.prev(m), n = c.next(m);
            float sv = 0.f;
            if (pm >= 0) sv = warp_pair_sim(c.row(pm), c.nrm(pm), c.row(n), c.nrm(n), C, lane);
            if (lane == 0) {
                c.kill(m, r);
                c.prev(n) = pm;
                if (pm >= 0) {
                    c.next(pm) = n;
                    c.sim(pm) = sv;
                    c.stamp(pm, r);
                }
            }
        }
        __syncthreads();
        return;
    }
    const int n = c.next(m), nd = c.n_dirty(r);
    if (tid == 0) s_cnt = 0;
    // ---- row tasks in batches of kBufs: task 0 = merge (m, n) -> m, task k > 0 = replay on dirty row k - 1
    for (int t0 = 0; t0 <= nd; t0 += kBufs) {
        if (tid < kBufs) s_changed[tid] = 0;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kBufs; ++k) {
            const int task = t0 + k;
            if (task > nd) break;
            const int j = task ? c.dirty(r, task - 1) : m;
            if (task && (j == m || j == n)) continue;
            const uint2* src = reinterpret_cast<const uint2*>(c.row(j));
            uint2* dst = reinterpret_cast<uint2*>(work_row(P, j, c.p));
            uint2* buf = reinterpret_cast<uint2*>(rowbuf + (size_t)k * C);
            if (task == 0) {
                const uint2* src2 = reinterpret_cast<const uint2*>(c.row(n));
                const float sa = c.size(m), sb = c.size(n);
                const float snew = round_bf16(sa + sb);
                for (int v0 = tid; v0 < nv; v0 += 4 * kMlThreads) {
                    uint2 q[4], w[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int v = v0 + u * kMlThreads;
                        if (v < nv) { q[u] = src[v]; w[u] = src2[v]; }
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int v = v0 + u * kMlThreads;
                        if (v < nv) {
                            uint2 y;
                            y.x = merge_pair(q[u].x, w[u].x, sa, sb, snew);
                            y.y = merge_pair(q[u].y, w[u].y, sa, sb, snew);
                            dst[v] = y;
                            buf[v] = y;
                        }
                    }
                }
                if (tid == 0) s_changed[k] = 1;
            } else {
                const float sz = c.size(j);
                bool diff = false;
                for (int v0 = tid; v0 < nv; v0 += 4 * kMlThreads) {
                    uint2 q[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int v = v0 + u * kMlThreads;
                        if (v < nv) q[u] = src[v];
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int v = v0 + u * kMlThreads;
                        if (v < nv) {
                            uint2 y;
                            y.x = rescale_pair(q[u].x, sz);
                            y.y = rescale_pair(q[u].y, sz);
                            diff |= (y.x != q[u].x) || (y.y != q[u].y);
                            dst[v] = y;
                            buf[v] = y;
                        }
                    }
                }
                if (diff) s_changed[k] = 1;
            }
        }
        __syncthreads();
        if (warp < kBufs && t0 + warp <= nd) {
            const int task = t0 + warp;
            const int j = task ? c.dirty(r, task - 1) : m;
            if (!(task && (j == m || j == n))) {
                const float nr = warp_row_norm(rowbuf + (size_t)warp * C, C, lane);
                if (lane == 0) {
                    c.nrm(j) = nr;
                    c.set_in_work(j);
                    if (s_changed[warp]) c.set_dirty(r + 1, atomicAdd(&s_cnt, 1), j);
                }
            }
        }
        __syncthreads();
    }
    if (tid == 0) {                                              // sizes and links: n leaves the list
        c.set_size(m, round_bf16(c.size(m) + c.size(n)));
        const int nx = c.next(n);
        c.next(m) = nx;
        if (nx < T) c.prev(nx) = m;
        c.kill(n, r);
    }
    __syncthreads();
    // ---- similarities on both sides of every changed row
    const int nch = s_cnt;
    for (int task = warp; task < 2 * nch; task += kMlWarps) {
        const int j = c.dirty(r + 1, task >> 1);
        int a, b;
        if (task & 1) { a = j; b = c.next(j); }
        else { a = c.prev(j); b = j; }
        if (a < 0) continue;
        float sv = -INFINITY;
        if (b < T) sv = warp_pair_sim(c.row(a), c.nrm(a), c.row(b), c.nrm(b), C, lane);
        if (lane == 0) {
            c.sim(a) = sv;
            c.stamp(a, r);
        }
    }
    c.end_round(r, nch);
    __syncthreads();
}

// sync mode, one round per launch: every patch merges or drops the frame of the shared argmax (merge_at[0], from
// mallm_sync_argmax_kernel); dynamic shared memory = the row buffers, kSyncBufs * C * 2 bytes (at most 32 KB)
constexpr int kSyncBufs = 2;
__global__ void __launch_bounds__(kMlThreads) mallm_round_kernel(MallmParams P, int round) {
    pdl_enter();
    extern __shared__ __align__(16) uint8_t smem_raw[];
    GlobalColumn c(P, blockIdx.x);
    mallm_round<kSyncBufs>(P, c, reinterpret_cast<__nv_bfloat16*>(smem_raw), round, P.merge_at[0]);
}

// patch-local mode: ALL rounds of one patch column in one CTA, the column state in shared memory (rounds_smem)
template <int kBufs>
__global__ void __launch_bounds__(kMlThreads) mallm_rounds_kernel(MallmParams P, int rounds) {
    pdl_enter();
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __shared__ Best s_best[kMlWarps];
    const int p = blockIdx.x, T = P.T;
    const RoundsSmem L = rounds_smem(T, P.C, kBufs);
    SmemColumn c{P, p,
                 reinterpret_cast<float*>(smem_raw + L.sim), reinterpret_cast<float*>(smem_raw + L.nrm),
                 reinterpret_cast<float*>(smem_raw + L.size), reinterpret_cast<int*>(smem_raw + L.next),
                 reinterpret_cast<int*>(smem_raw + L.prev), reinterpret_cast<short*>(smem_raw + L.dirty),
                 smem_raw + L.in_work, P.hard ? 0 : P.n_dirty[p]};
    for (int i = threadIdx.x; i < T; i += blockDim.x) {
        const size_t a = at(P, i, p);
        c.sim_[i] = P.sim[a];
        c.nrm_[i] = P.nrm[a];
        c.next_[i] = P.next[a];
        c.prev_[i] = P.prev[a];
        if (!P.hard) {
            c.size_[i] = P.size[a];
            c.in_work_[i] = P.in_work[a];
        }
    }
    for (int k = threadIdx.x; k < c.nd; k += blockDim.x) c.set_dirty(0, k, P.dirty[(size_t)p * T + k]);
    __syncthreads();
    __nv_bfloat16* rowbuf = reinterpret_cast<__nv_bfloat16*>(smem_raw + L.rowbuf);
    for (int r = 0; r < rounds; ++r) mallm_round<kBufs>(P, c, rowbuf, r, block_argmax(c.sim_, 1, T, s_best));
}

// ------------------------------------------------------------------------------------- sync mode: mean + argmax
// ATen's bf16 mean(-1) over n contiguous values (held as fp32), times fp32(1/n) and rounded by the caller.
// `shift` = (byte offset of the row in the reference's bf16 tensor % 16) / 2.  Result valid in lane 0.
__device__ __forceinline__ float aten_row_sum_bf16(const float* __restrict__ row, int n, int shift, int lane) {
    float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    int width = 1, nacc = 8;
    if (n >= 128) {
        while (width * 2 <= (n >> 3) && width < 32) width *= 2;
        int start = 0;
        if (shift > 0) {
            if (lane >= shift && lane < 8) a[0] += row[lane - shift];
            start = 8 - shift;
        }
        const int body = (n - start) >> 3;
        if (lane < width)
            for (int idx = lane; idx < body; idx += width) {
                const float* q = row + start + idx * 8;
#pragma unroll
                for (int j = 0; j < 8; ++j) a[j] += q[j];
            }
        const int tail = start + body * 8 + lane;
        if (tail < n) a[0] += row[tail];
    } else {
        nacc = 4;
        while (width * 2 <= n && width < 32) width *= 2;
        if (lane < width) {
            int k = 0;
            for (int idx = lane; idx < n; idx += width, k = (k + 1) & 3) a[k] += row[idx];
        }
    }
    float s = ((a[0] + a[1]) + a[2]) + a[3];
    if (nacc == 8) s = (((s + a[4]) + a[5]) + a[6]) + a[7];
    for (int off = width >> 1; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
    return s;
}

// Block-wide exclusive count of the surviving frames of patch p.  Each thread owns one chunk [i0, i1) of
// ceil(T / blockDim.x) frames, in thread order; the result is the number of survivors before i0.  `warp_tot`: 32 ints.
__device__ __forceinline__ int alive_before(const MallmParams& P, int p, int& i0, int& i1, int* warp_tot) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int per = (P.T + blockDim.x - 1) / blockDim.x;
    i0 = threadIdx.x * per;
    i1 = min(P.T, i0 + per);
    int cnt = 0;
    for (int i = i0; i < i1; ++i) cnt += P.alive[at(P, i, p)];
    int inc = cnt;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += o;
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int t = (lane < nw) ? warp_tot[lane] : 0;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int o = __shfl_up_sync(0xffffffffu, t, off);
            if (lane >= off) t += o;
        }
        warp_tot[lane] = t;
    }
    __syncthreads();
    return inc - cnt + (warp ? warp_tot[warp - 1] : 0);
}

// one CTA: refresh the mean similarity of the rows rewritten in the round stamped `stamp` (all rows when the row
// alignment depends on the position, i.e. N % 8 != 0), then the shared argmax
__global__ void __launch_bounds__(1024) mallm_sync_argmax_kernel(MallmParams P, int stamp) {
    pdl_enter();
    extern __shared__ __align__(16) uint8_t smem_raw[];
    int* pos = reinterpret_cast<int*>(smem_raw);                 // [T] index of frame i among the survivors
    __shared__ int s_warp_tot[32];
    __shared__ Best s_best[32];
    const int T = P.T, N = P.N;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const bool all = (N & 7) != 0 || stamp == 0;
    if (all && N >= 128 && (N & 7)) {
        int i0, i1;
        int run = alive_before(P, 0, i0, i1, s_warp_tot);
        for (int i = i0; i < i1; ++i) {
            pos[i] = run;
            run += P.alive[at(P, i, 0)];
        }
        __syncthreads();
    }
    const float rcp = 1.0f / (float)N;
    // rows whose mean has to be refreshed: all of them, or the (few) rows stamped by this round's merge kernels - the
    // stamps are fetched by all threads at once and compacted into a task list, one warp per task
    __shared__ int s_ntask;
    int* tasks = pos + T;                                        // [T]
    if (threadIdx.x == 0) s_ntask = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < T; i += blockDim.x)
        if (all || P.touched[i] == stamp) tasks[atomicAdd(&s_ntask, 1)] = i;
    __syncthreads();
    const int ntask = s_ntask;
    for (int k = warp; k < ntask; k += nw) {
        const int i = tasks[k];
        const float* row = P.sim + (size_t)i * P.si;
        float v = -INFINITY;
        if (row[0] != -INFINITY) {                               // dead and last rows hold -inf in every patch
            const int shift = (N >= 128 && (N & 7)) ? (int)(((long long)pos[i] * N) & 7) : 0;
            v = round_bf16(aten_row_sum_bf16(row, N, shift, lane) * rcp);
        }
        if (lane == 0) P.msim[i] = v;
    }
    __syncthreads();
    const int m = block_argmax(P.msim, 1, T, s_best);
    if (threadIdx.x == 0) P.merge_at[0] = m;
}

// --------------------------------------------------------------------------------------------- compaction
// one CTA per patch: surviving rows in frame order -> out[pos, p, :], sizes_out[pos, p]
__global__ void __launch_bounds__(kMlThreads) mallm_emit_kernel(MallmParams P, __nv_bfloat16* __restrict__ out,
                                                               __nv_bfloat16* __restrict__ sizes_out, int t) {
    pdl_enter();
    extern __shared__ __align__(16) uint8_t smem_raw[];
    int* order = reinterpret_cast<int*>(smem_raw);               // [t]
    __shared__ int s_warp_tot[32];
    const int p = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const GlobalColumn c(P, p);
    int i0, i1;
    int base = alive_before(P, p, i0, i1, s_warp_tot);
    for (int i = i0; i < i1; ++i)
        if (P.alive[at(P, i, p)]) {
            if (base < t) order[base] = i;
            ++base;
        }
    __syncthreads();
    const int nvec = P.C >> 3;
    for (int j = warp; j < t; j += kMlWarps) {
        const int i = order[j];
        const uint4* src = reinterpret_cast<const uint4*>(c.row(i));
        uint4* dst = reinterpret_cast<uint4*>(out + ((size_t)j * P.N + p) * (size_t)P.C);
        int v = lane;
        for (; v + (kBatch - 1) * 32 < nvec; v += kBatch * 32) {
            uint4 b[kBatch];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) b[u] = src[v + 32 * u];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) dst[v + 32 * u] = b[u];
        }
        for (; v < nvec; v += 32) dst[v] = src[v];
        if (lane == 0 && sizes_out) sizes_out[(size_t)j * P.N + p] = __float2bfloat16_rn(c.size(i));
    }
}

static size_t align_up(size_t v) { return (v + 255) & ~(size_t)255; }

struct MallmLayout {
    size_t sim, nrm, size, next, prev, alive, in_work, dirty, n_dirty, merge_at, msim, touched, work, total;
};
static MallmLayout mallm_layout(int64_t T, int64_t N, int64_t C, int hard) {
    MallmLayout L;
    const size_t tn = (size_t)T * N;
    size_t o = 0;
    L.sim = o; o = align_up(o + tn * 4);
    L.nrm = o; o = align_up(o + tn * 4);
    L.size = o; o = align_up(o + tn * 4);
    L.next = o; o = align_up(o + tn * 4);
    L.prev = o; o = align_up(o + tn * 4);
    L.alive = o; o = align_up(o + tn);
    L.in_work = o; o = align_up(o + tn);
    L.dirty = o; o = align_up(o + 2 * tn * 4);
    L.n_dirty = o; o = align_up(o + 2 * (size_t)N * 4);
    L.merge_at = o; o = align_up(o + 4);
    L.msim = o; o = align_up(o + (size_t)T * 4);
    L.touched = o; o = align_up(o + (size_t)T * 4);
    L.work = o; o = align_up(o + (hard ? 0 : tn * (size_t)C * 2));
    L.total = o;
    return L;
}

}  // namespace rtk

using namespace rtk;

extern "C" size_t rtk_mallm_workspace_bytes(int64_t T, int64_t N, int64_t C, int hard) {
    if (T <= 0 || N <= 0 || C <= 0) return 0;
    return mallm_layout(T, N, C, hard).total;
}

extern "C" int rtk_mallm_compress(const void* x, const void* sizes_in, int64_t T, int64_t N, int64_t C, int64_t t, int sync,
                                  int hard, void* out, void* sizes_out, void* workspace, size_t workspace_bytes,
                                  void* stream_) {
    RTK_NVTX("rtk_mallm_compress");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!x || !out || !workspace || T < 1 || N < 1 || t < 1 || t > T) return RTK_E_BADARG;
    if (C % 8 != 0 || C < 256 || C > 8192 || T > 8192 || N > 65535) return RTK_E_UNSUPPORTED;
    if (((uintptr_t)x | (uintptr_t)out | (uintptr_t)workspace) & 15u) return RTK_E_ALIGN;
    const MallmLayout L = mallm_layout(T, N, C, hard);
    if (workspace_bytes < L.total) return RTK_E_WORKSPACE;
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    MallmParams P;
    P.x = static_cast<const __nv_bfloat16*>(x);
    P.work = reinterpret_cast<__nv_bfloat16*>(ws + L.work);
    P.sizes_in = static_cast<const __nv_bfloat16*>(sizes_in);
    P.T = (int)T; P.N = (int)N; P.C = (int)C;
    // the shared argmax of sync mode reads one frame across patches, the per-patch argmax one patch across frames
    P.si = sync ? N : 1;
    P.sp = sync ? 1 : T;
    P.sim = reinterpret_cast<float*>(ws + L.sim);
    P.nrm = reinterpret_cast<float*>(ws + L.nrm);
    P.size = reinterpret_cast<float*>(ws + L.size);
    P.next = reinterpret_cast<int*>(ws + L.next);
    P.prev = reinterpret_cast<int*>(ws + L.prev);
    P.alive = ws + L.alive;
    P.in_work = ws + L.in_work;
    P.dirty = reinterpret_cast<int*>(ws + L.dirty);
    P.n_dirty = reinterpret_cast<int*>(ws + L.n_dirty);
    P.merge_at = reinterpret_cast<int*>(ws + L.merge_at);
    P.msim = reinterpret_cast<float*>(ws + L.msim);
    P.touched = reinterpret_cast<int*>(ws + L.touched);
    P.sync = sync ? 1 : 0;
    P.hard = hard ? 1 : 0;
    const int rounds = (int)(T - t);
    const size_t scan_smem = (size_t)T * 8;                     // positions + task list of the sync argmax kernel
    const size_t row_smem = hard ? 0 : (size_t)kSyncBufs * C * 2;   // row buffers of the sync round kernel, <= 32 KB
    const size_t emit_smem = (size_t)t * 4;
    void (*rounds_kernel)(MallmParams, int) = mallm_rounds_kernel<2>;
    size_t rounds_bytes = 0;
    cudaError_t e;
    if (!sync && rounds > 0) {
        // the per-patch state in shared memory, with two row buffers when they fit (1 KB is left for the kernel's
        // static shared memory); one buffer fits up to T = C = 8192 on a B200
        int dev = 0, optin = 0;
        if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
        if ((e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return (int)e;
        const int bufs = rounds_smem((int)T, (int)C, 2).bytes + 1024 <= (size_t)optin ? 2 : 1;
        rounds_bytes = rounds_smem((int)T, (int)C, bufs).bytes;
        if (rounds_bytes + 1024 > (size_t)optin) return RTK_E_UNSUPPORTED;
        if (bufs == 1) rounds_kernel = mallm_rounds_kernel<1>;
        e = cudaFuncSetAttribute(rounds_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rounds_bytes);
        if (e != cudaSuccess) return (int)e;
    }
    if (sync) {
        e = cudaFuncSetAttribute(mallm_sync_argmax_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_smem);
        if (e != cudaSuccess) return (int)e;
    }
    e = cudaFuncSetAttribute(mallm_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)emit_smem);
    if (e != cudaSuccess) return (int)e;
    if (T >= 2) {
        const int rc = dpselect_sim_nrm(x, T, N, C, DisAux{P.sim, P.nrm, P.si, P.sp}, stream);
        if (rc) return rc;
    }
    RTK_LAUNCH_PDL(mallm_init_kernel, (unsigned)N, kMlThreads, 0, stream, P);
    if (!sync) {
        if (rounds > 0) RTK_LAUNCH_PDL(rounds_kernel, (unsigned)N, kMlThreads, rounds_bytes, stream, P, rounds);
    } else {
        for (int r = 0; r < rounds; ++r) {
            RTK_LAUNCH_PDL(mallm_sync_argmax_kernel, 1, 1024, scan_smem, stream, P, r);
            RTK_LAUNCH_PDL(mallm_round_kernel, (unsigned)N, kMlThreads, row_smem, stream, P, r);
        }
    }
    RTK_LAUNCH_PDL(mallm_emit_kernel, (unsigned)N, kMlThreads, emit_smem, stream, P, static_cast<__nv_bfloat16*>(out), hard ? nullptr : static_cast<__nv_bfloat16*>(sizes_out), (int)t);
    return 0;
}
