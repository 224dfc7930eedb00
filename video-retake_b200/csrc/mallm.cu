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
//   * patch-local mode runs all rounds of a patch column inside one CTA of one launch; sync mode shares one argmax
//     over the bf16 mean of the similarities across patches (one round kernel + one argmax kernel per round).
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

__device__ __forceinline__ const __nv_bfloat16* row_ptr(const MallmParams& P, int i, int p) {
    const size_t off = ((size_t)i * P.N + p) * (size_t)P.C;
    return (!P.hard && P.in_work[at(P, i, p)]) ? P.work + off : P.x + off;
}

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

// soft merge of frames m and next(m) of patch p by the whole CTA; `round` = number of merges already done;
// simv[i * sstride] is the patch's similarity column (global state, or the shared-memory copy of the persistent loop)
__device__ __forceinline__ void mallm_soft_round(const MallmParams& P, int p, int round, int m, float* simv, long long sstride) {
    __shared__ int s_n, s_cnt;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int T = P.T, C = P.C;
    if (threadIdx.x == 0) {
        s_n = P.next[at(P, m, p)];
        s_cnt = 0;
    }
    __syncthreads();
    const int n = s_n;
    const int* cur = P.dirty + ((size_t)(round & 1) * P.N + p) * T;
    int* nxt = P.dirty + ((size_t)((round + 1) & 1) * P.N + p) * T;
    const int nd = P.n_dirty[(size_t)(round & 1) * P.N + p];
    const size_t row_elems = (size_t)C;
    // ---- row tasks: task 0 merges (m, n) into m; task k > 0 replays x = rd(rd(x * s) / s) on a dirty row
    for (int task = warp; task <= nd; task += kMlWarps) {
        const int j = task ? cur[task - 1] : m;
        if (task && (j == m || j == n)) continue;
        const size_t a = at(P, j, p);
        const uint2* src = reinterpret_cast<const uint2*>(row_ptr(P, j, p));
        uint2* dst = reinterpret_cast<uint2*>(P.work + ((size_t)j * P.N + p) * row_elems);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        bool changed = true;
        const int nv = C >> 2;
        if (task == 0) {
            const uint2* src2 = reinterpret_cast<const uint2*>(row_ptr(P, n, p));
            const float sa = P.size[a], sb = P.size[at(P, n, p)];
            const float snew = round_bf16(sa + sb);
            auto step = [&](int v, const uint2& q, const uint2& r) {
                uint2 y;
                y.x = merge_pair(q.x, r.x, sa, sb, snew);
                y.y = merge_pair(q.y, r.y, sa, sb, snew);
                dst[v] = y;
                fma_sq_bf16x2(a0, a1, y.x);
                fma_sq_bf16x2(a2, a3, y.y);
            };
            constexpr int kHalf = kBatch / 2;
            int v = lane;
            for (; v + (kHalf - 1) * 32 < nv; v += kHalf * 32) {
                uint2 q[kHalf], r[kHalf];
#pragma unroll
                for (int u = 0; u < kHalf; ++u) { q[u] = src[v + 32 * u]; r[u] = src2[v + 32 * u]; }
#pragma unroll
                for (int u = 0; u < kHalf; ++u) step(v + 32 * u, q[u], r[u]);
            }
            for (; v < nv; v += 32) step(v, src[v], src2[v]);
            if (lane == 0) P.size[a] = snew;
        } else {
            const float s = P.size[a];
            bool diff = false;
            auto step = [&](int v, const uint2& q) {
                uint2 y;
                y.x = rescale_pair(q.x, s);
                y.y = rescale_pair(q.y, s);
                diff |= (y.x != q.x) || (y.y != q.y);
                dst[v] = y;
                fma_sq_bf16x2(a0, a1, y.x);
                fma_sq_bf16x2(a2, a3, y.y);
            };
            int v = lane;
            for (; v + (kBatch - 1) * 32 < nv; v += kBatch * 32) {
                uint2 q[kBatch];
#pragma unroll
                for (int u = 0; u < kBatch; ++u) q[u] = src[v + 32 * u];
#pragma unroll
                for (int u = 0; u < kBatch; ++u) step(v + 32 * u, q[u]);
            }
            for (; v < nv; v += 32) step(v, src[v]);
            changed = __any_sync(0xffffffffu, diff);
        }
        const float nr = clamp_norm(warp_tree(((a0 + a1) + a2) + a3, lane));
        if (lane == 0) {
            P.nrm[a] = nr;
            P.in_work[a] = 1;
            if (changed) nxt[atomicAdd(&s_cnt, 1)] = j;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {                                      // unlink n
        const int nx = P.next[at(P, n, p)];
        P.next[at(P, m, p)] = nx;
        if (nx < T) P.prev[at(P, nx, p)] = m;
        P.alive[at(P, n, p)] = 0;
        simv[(size_t)n * sstride] = -INFINITY;
        if (P.sync && p == 0) P.touched[n] = round + 1;
        P.n_dirty[(size_t)((round + 1) & 1) * P.N + p] = s_cnt;
    }
    __syncthreads();
    // ---- similarities on both sides of every changed row
    const int nch = s_cnt;
    for (int task = warp; task < 2 * nch; task += kMlWarps) {
        const int j = nxt[task >> 1];
        int a, b;
        if (task & 1) { a = j; b = P.next[at(P, j, p)]; }
        else { a = P.prev[at(P, j, p)]; b = j; }
        if (a < 0) continue;
        float s = -INFINITY;
        if (b < T) s = warp_pair_sim(row_ptr(P, a, p), P.nrm[at(P, a, p)], row_ptr(P, b, p), P.nrm[at(P, b, p)], C, lane);
        if (lane == 0) {
            simv[(size_t)a * sstride] = s;
            if (P.sync) P.touched[a] = round + 1;
        }
    }
}

// hard variant: frame m is deleted, nothing is rewritten (one warp's work)
__device__ __forceinline__ void mallm_hard_round(const MallmParams& P, int p, int round, int m, float* simv, long long sstride) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp != 0) return;
    const int pm = P.prev[at(P, m, p)], n = P.next[at(P, m, p)];
    float s = 0.f;
    if (pm >= 0) s = warp_pair_sim(row_ptr(P, pm, p), P.nrm[at(P, pm, p)], row_ptr(P, n, p), P.nrm[at(P, n, p)], P.C, lane);
    if (lane == 0) {
        P.alive[at(P, m, p)] = 0;
        simv[(size_t)m * sstride] = -INFINITY;
        P.prev[at(P, n, p)] = pm;
        if (pm >= 0) {
            P.next[at(P, pm, p)] = n;
            simv[(size_t)pm * sstride] = s;
        }
        if (P.sync && p == 0) {
            P.touched[m] = round + 1;
            if (pm >= 0) P.touched[pm] = round + 1;
        }
    }
}

// one round per launch (sync mode: the shared argmax comes from mallm_sync_argmax_kernel of the previous launch)
__global__ void __launch_bounds__(kMlThreads) mallm_round_kernel(MallmParams P, int round) {
    pdl_enter();
    __shared__ Best s_best[kMlWarps];
    const int p = blockIdx.x;
    float* simv = P.sim + (size_t)p * P.sp;
    const int m = P.sync ? P.merge_at[0] : block_argmax(simv, P.si, P.T, s_best);
    if (P.hard) mallm_hard_round(P, p, round, m, simv, P.si);
    else mallm_soft_round(P, p, round, m, simv, P.si);
}

// patch-local mode: ALL rounds of one patch column in one CTA, the similarity column lives in shared memory
__global__ void __launch_bounds__(kMlThreads) mallm_rounds_kernel(MallmParams P, int rounds) {
    pdl_enter();
    extern __shared__ __align__(16) uint8_t smem_raw[];
    float* sim_s = reinterpret_cast<float*>(smem_raw);           // [T]
    __shared__ Best s_best[kMlWarps];
    const int p = blockIdx.x;
    for (int i = threadIdx.x; i < P.T; i += blockDim.x) sim_s[i] = P.sim[at(P, i, p)];
    __syncthreads();
    for (int r = 0; r < rounds; ++r) {
        const int m = block_argmax(sim_s, 1, P.T, s_best);
        if (P.hard) mallm_hard_round(P, p, r, m, sim_s, 1);
        else mallm_soft_round(P, p, r, m, sim_s, 1);
        __syncthreads();
    }
}


// Patch-local mode, fast variant: the whole per-patch state (similarities, norms, sizes, links, flags, dirty lists)
// lives in shared memory for all rounds, and the row work of a round is done by the whole CTA: the merge (and the
// replay on dirty rows) is element-wise over 256 threads with every load of the round in flight at once, the result
// goes to the workspace row AND to a shared-memory row buffer from which ONE warp then takes the norm in ATen's order.
// Only `alive`, `in_work`, `size` (read by the emit kernel) and the rewritten rows go back to global memory.
constexpr int kRowBufs = 2;      // row tasks handled per batch (merge + one dirty row is the common case)

struct RoundsSmem {
    float *sim, *nrm, *size;
    int *next, *prev;
    short* dirty;                // [2][T]
    uint8_t* in_work;
    __nv_bfloat16* rowbuf;       // [kRowBufs][C]
};
__host__ __device__ inline size_t rounds_smem_bytes(int T, int C) {
    return (size_t)T * (5 * 4 + 2 * 2 + 1) + 16 + (size_t)kRowBufs * C * 2 + 16;
}

__global__ void __launch_bounds__(kMlThreads) mallm_rounds_smem_kernel(MallmParams P, int rounds) {
    pdl_enter();
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __shared__ Best s_best[kMlWarps];
    __shared__ int s_cnt, s_changed[kRowBufs];
    const int p = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int T = P.T, C = P.C, nv = C >> 2;
    RoundsSmem S;
    {
        uint8_t* q = smem_raw;
        S.sim = reinterpret_cast<float*>(q);   q += (size_t)T * 4;
        S.nrm = reinterpret_cast<float*>(q);   q += (size_t)T * 4;
        S.size = reinterpret_cast<float*>(q);  q += (size_t)T * 4;
        S.next = reinterpret_cast<int*>(q);    q += (size_t)T * 4;
        S.prev = reinterpret_cast<int*>(q);    q += (size_t)T * 4;
        S.dirty = reinterpret_cast<short*>(q); q += (size_t)T * 4;
        S.in_work = q;                         q += ((size_t)T + 15) & ~(size_t)15;
        S.rowbuf = reinterpret_cast<__nv_bfloat16*>(q);
    }
    for (int i = tid; i < T; i += blockDim.x) {
        const size_t a = at(P, i, p);
        S.sim[i] = P.sim[a];
        S.nrm[i] = P.nrm[a];
        S.next[i] = P.next[a];
        S.prev[i] = P.prev[a];
        if (!P.hard) {
            S.size[i] = P.size[a];
            S.in_work[i] = P.in_work[a];
        }
    }
    int nd = 0;
    if (!P.hard) {
        nd = P.n_dirty[p];
        for (int i = tid; i < nd; i += blockDim.x) S.dirty[i] = (short)P.dirty[(size_t)p * T + i];
    }
    __syncthreads();
    auto row = [&](int i) -> const __nv_bfloat16* {
        const size_t off = ((size_t)i * P.N + p) * (size_t)C;
        return (!P.hard && S.in_work[i]) ? P.work + off : P.x + off;
    };
    for (int r = 0; r < rounds; ++r) {
        const int m = block_argmax(S.sim, 1, T, s_best);
        if (P.hard) {
            if (warp == 0) {
                const int pm = S.prev[m], n = S.next[m];
                float sv = 0.f;
                if (pm >= 0) sv = warp_pair_sim(row(pm), S.nrm[pm], row(n), S.nrm[n], C, lane);
                if (lane == 0) {
                    P.alive[at(P, m, p)] = 0;
                    S.sim[m] = -INFINITY;
                    S.prev[n] = pm;
                    if (pm >= 0) {
                        S.next[pm] = n;
                        S.sim[pm] = sv;
                    }
                }
            }
            __syncthreads();
            continue;
        }
        const int n = S.next[m];
        const short* cur = S.dirty + (size_t)(r & 1) * T;
        short* nxt = S.dirty + (size_t)((r + 1) & 1) * T;
        if (tid == 0) s_cnt = 0;
        // ---- row tasks in batches of kRowBufs: task 0 = merge (m, n) -> m, task k > 0 = replay on dirty row cur[k - 1]
        for (int t0 = 0; t0 <= nd; t0 += kRowBufs) {
            if (tid < kRowBufs) s_changed[tid] = 0;
            __syncthreads();
#pragma unroll
            for (int k = 0; k < kRowBufs; ++k) {
                const int task = t0 + k;
                if (task > nd) break;
                const int j = task ? cur[task - 1] : m;
                if (task && (j == m || j == n)) continue;
                const uint2* src = reinterpret_cast<const uint2*>(row(j));
                uint2* dst = reinterpret_cast<uint2*>(P.work + ((size_t)j * P.N + p) * (size_t)C);
                uint2* buf = reinterpret_cast<uint2*>(S.rowbuf + (size_t)k * C);
                if (task == 0) {
                    const uint2* src2 = reinterpret_cast<const uint2*>(row(n));
                    const float sa = S.size[m], sb = S.size[n];
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
                    const float sz = S.size[j];
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
            if (warp < kRowBufs && t0 + warp <= nd) {
                const int task = t0 + warp;
                const int j = task ? cur[task - 1] : m;
                if (!(task && (j == m || j == n))) {
                    const float nr = warp_row_norm(S.rowbuf + (size_t)warp * C, C, lane);
                    if (lane == 0) {
                        S.nrm[j] = nr;
                        S.in_work[j] = 1;
                        P.in_work[at(P, j, p)] = 1;
                        if (s_changed[warp]) nxt[atomicAdd(&s_cnt, 1)] = (short)j;
                    }
                }
            }
            __syncthreads();
        }
        if (tid == 0) {                                          // sizes and links
            const float snew = round_bf16(S.size[m] + S.size[n]);
            S.size[m] = snew;
            P.size[at(P, m, p)] = snew;
            const int nx = S.next[n];
            S.next[m] = nx;
            if (nx < T) S.prev[nx] = m;
            P.alive[at(P, n, p)] = 0;
            S.sim[n] = -INFINITY;
        }
        __syncthreads();
        // ---- similarities on both sides of every changed row
        const int nch = s_cnt;
        for (int task = warp; task < 2 * nch; task += kMlWarps) {
            const int j = nxt[task >> 1];
            int a, b;
            if (task & 1) { a = j; b = S.next[j]; }
            else { a = S.prev[j]; b = j; }
            if (a < 0) continue;
            float sv = -INFINITY;
            if (b < T) sv = warp_pair_sim(row(a), S.nrm[a], row(b), S.nrm[b], C, lane);
            if (lane == 0) S.sim[a] = sv;
        }
        nd = nch;
        __syncthreads();
    }
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
        // exclusive scan of the alive flags, chunk per thread
        const int per = (T + blockDim.x - 1) / blockDim.x;
        const int i0 = threadIdx.x * per, i1 = min(T, i0 + per);
        int cnt = 0;
        for (int i = i0; i < i1; ++i) cnt += P.alive[at(P, i, 0)];
        int inc = cnt;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int o = __shfl_up_sync(0xffffffffu, inc, off);
            if (lane >= off) inc += o;
        }
        if (lane == 31) s_warp_tot[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            int t = (lane < nw) ? s_warp_tot[lane] : 0;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const int o = __shfl_up_sync(0xffffffffu, t, off);
                if (lane >= off) t += o;
            }
            s_warp_tot[lane] = t;
        }
        __syncthreads();
        int run = inc - cnt + (warp ? s_warp_tot[warp - 1] : 0);
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
    __shared__ int s_warp_tot[kMlWarps];
    const int p = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int T = P.T;
    const int per = (T + kMlThreads - 1) / kMlThreads;
    const int i0 = threadIdx.x * per, i1 = min(T, i0 + per);
    int cnt = 0;
    for (int i = i0; i < i1; ++i) cnt += P.alive[at(P, i, p)];
    int inc = cnt;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += o;
    }
    if (lane == 31) s_warp_tot[warp] = inc;
    __syncthreads();
    int base = inc - cnt;
    for (int w = 0; w < warp; ++w) base += s_warp_tot[w];
    for (int i = i0; i < i1; ++i)
        if (P.alive[at(P, i, p)]) {
            if (base < t) order[base] = i;
            ++base;
        }
    __syncthreads();
    const int nvec = P.C >> 3;
    for (int j = warp; j < t; j += kMlWarps) {
        const int i = order[j];
        const uint4* src = reinterpret_cast<const uint4*>(row_ptr(P, i, p));
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
        if (lane == 0 && sizes_out) sizes_out[(size_t)j * P.N + p] = __float2bfloat16_rn(P.size[at(P, i, p)]);
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
    const size_t scan_smem = (size_t)T * 8;                     // positions + task list of the sync argmax kernel
    if (sync) {
        cudaError_t e = cudaFuncSetAttribute(mallm_sync_argmax_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_smem);
        if (e != cudaSuccess) return (int)e;
    }
    if (T >= 2) {
        const int rc = dpselect_sim_nrm(x, T, N, C, DisAux{P.sim, P.nrm, P.si, P.sp}, stream);
        if (rc) return rc;
    }
    RTK_LAUNCH_PDL(mallm_init_kernel, (unsigned)N, kMlThreads, 0, stream, P);
    if (sync && t < T) {
        RTK_LAUNCH_PDL(mallm_sync_argmax_kernel, 1, 1024, scan_smem, stream, P, 0);
    }
    const int rounds = (int)(T - t);
    if (!sync) {
        if (rounds > 0) {
            int dev = 0, smem_max = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
            const size_t need = rounds_smem_bytes((int)T, (int)C);
            if (need + 1024 <= (size_t)smem_max) {                 // whole per-patch state in shared memory
                cudaError_t e2 = cudaFuncSetAttribute(mallm_rounds_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need);
                if (e2 != cudaSuccess) return (int)e2;
                RTK_LAUNCH_PDL(mallm_rounds_smem_kernel, (unsigned)N, kMlThreads, need, stream, P, rounds);
            } else {                                              // very long videos: state stays in global memory
                // only the similarity column lives in shared memory: T floats, at most 32 KB, under the 48 KB default
                RTK_LAUNCH_PDL(mallm_rounds_kernel, (unsigned)N, kMlThreads, (size_t)T * 4, stream, P, rounds);
            }
        }
    } else {
        for (int r = 0; r < rounds; ++r) {
            RTK_LAUNCH_PDL(mallm_round_kernel, (unsigned)N, kMlThreads, 0, stream, P, r);
            if (r + 1 < rounds) {
                RTK_LAUNCH_PDL(mallm_sync_argmax_kernel, 1, 1024, scan_smem, stream, P, r + 1);
            }
        }
    }
    const size_t emit_smem = (size_t)t * 4;
    cudaError_t e = cudaFuncSetAttribute(mallm_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)emit_smem);
    if (e != cudaSuccess) return (int)e;
    RTK_LAUNCH_PDL(mallm_emit_kernel, (unsigned)N, kMlThreads, emit_smem, stream, P, static_cast<__nv_bfloat16*>(out), hard ? nullptr : static_cast<__nv_bfloat16*>(sizes_out), (int)t);
    return 0;
}
