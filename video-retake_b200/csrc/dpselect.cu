// DPSelect kernels (sm_100a): adjacent-frame cosine distance, peak/top-t selection, row compaction.
// Replaces the torch op sequence of retake/visual_compression.py:98-177 (memory_bank_compress_keyframe).
//
// A1  dpselect_dis_kernel     HBM-bound.  Each warp owns one patch column p over a run of frames and streams
//     the 2*C-byte rows x[f, p, :] through a private shared-memory ring filled by 1-D TMA bulk copies
//     (cp.async.bulk + mbarrier), so every row is read from HBM exactly once (plus one halo row per run)
//     and the loads of the next rows are in flight while the current one is reduced.  The arithmetic replays
//     ATen-CUDA's F.cosine_similarity on bf16 bit for bit (tests/probes/probe_aten_cuda2.py):
//       n   = bf16(sqrt(sum_f32 x^2))        reduction order of Reduce.cuh with 4-element vectors
//       u_i = bf16(x_i / max(n, bf16(1e-8))) (computed as x_i * rcp(n): same bf16 result, see DESIGN.md)
//       p_i = bf16(u_i * w_i)
//       sim = bf16(sum_f32 p_i)              reduction order of Reduce.cuh with 8-element vectors
//       dis = 1 - float(sim)
//     Both orders are produced from ONE register layout (lane l holds the 4-element vectors l, l+32, ...).
// A2  dpselect_select_kernel  latency-bound (<= a few MB).  Warp per patch column held in shared memory: peaks,
//     key = dis + 2*peak, bitwise descent for the t-th largest radix key, ordered emission with ATen's tie rule.
// A3  dpselect_gather_kernel  HBM-bound row gather (stream compaction of surviving tokens).
#include <climits>

#include "rtk_common.cuh"

namespace rtk {

// ============================================================================================ A1: distance
#ifndef RTK_DIS_WARPS
#define RTK_DIS_WARPS 8
#endif
constexpr int kDisWarps = RTK_DIS_WARPS;
constexpr int kDisThreads = kDisWarps * kWarp;

struct RowCursor {
    // iterates the rows one warp has to read: items i = first, first+stride, ...; item -> (run, p);
    // run r covers computed frames [1 + r*R, min(1 + (r+1)*R, T)) and reads rows [r*R, that end).
    int item, stride, n_items, N, R, T;
    int p, f, fbeg, fend;
    __device__ __forceinline__ void load() {
        if (item < n_items) {
            int run = item / N;
            p = item - run * N;
            fbeg = run * R;
            fend = min(1 + (run + 1) * R, T);
            f = fbeg;
        }
    }
    __device__ __forceinline__ void init(int first, int stride_, int n_items_, int N_, int R_, int T_) {
        item = first; stride = stride_; n_items = n_items_; N = N_; R = R_; T = T_;
        load();
    }
    __device__ __forceinline__ bool valid() const { return item < n_items; }
    __device__ __forceinline__ void advance() {
        if (++f >= fend) { item += stride; load(); }
    }
};

// short rows (K4 <= 16, <= 120 registers) run two CTAs per SM so that 16 warps hide the per-row reduction latency
template <int K4, bool AUX, bool EXACT>   // EXACT: C == K4 * 128, every lane owns K4 full vectors (no bounds checks)
__global__ void __launch_bounds__(kDisThreads, (K4 <= 16) ? 2 : 1)
dpselect_dis_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ dis, int T, int N, int C, int R,
                    int n_items, int stages, int halo, DisAux aux, int active) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t row_bytes = (uint32_t)C * 2u;
    const int nv4 = C >> 2;                                  // 4-element vectors per row
    uint8_t* ring = smem + (size_t)warp * stages * row_bytes;
    const uint32_t ring_u32 = smem_u32(ring);
    const uint32_t bars = smem_u32(smem + (size_t)active * stages * row_bytes) + (uint32_t)(warp * stages) * 8u;

    if (lane == 0) {
        for (int s = 0; s < stages; ++s) mbar_init(bars + 8u * s, 1);
        fence_mbar_init();
    }
    __syncthreads();

    // rows longer than 7 KB leave room for fewer than two ring stages per warp with eight warps: then only `active`
    // warps of the CTA stream rows (the rest idle after the barrier above)
    if (warp >= active) return;
    const int gw = blockIdx.x * active + warp;
    const int GW = gridDim.x * active;
    RowCursor cons, prod;
    cons.init(gw, GW, n_items, N, R, T);
    prod = cons;

    auto issue = [&](const RowCursor& c, int s) {
        const __nv_bfloat16* src = x + ((size_t)c.f * N + c.p) * (size_t)C;
        mbar_arrive_expect_tx(bars + 8u * s, row_bytes);
        bulk_g2s(ring_u32 + (uint32_t)s * row_bytes, src, row_bytes, bars + 8u * s);
    };
    if (lane == 0) {
        for (int s = 0; s < stages && prod.valid(); ++s) { issue(prod, s); prod.advance(); }
    }

    const float eps = __uint_as_float(0x322c0000u);          // bf16(1e-8) widened (clamp_min_ on a bf16 tensor)
    int consumed = 0;
    // one row: wait for its bytes, reduce the norm, refill the ring slot, normalise into `cur`, and (unless it is the
    // first row of an item) emit the distance against `prev`.  Called with the two register files swapped on
    // alternate rows so that "previous row" never has to be copied.
    auto process_row = [&](uint2 (&cur)[K4], const uint2 (&prev)[K4]) {
        const int s = consumed % stages;
        mbar_wait(bars + 8u * s, (uint32_t)(consumed / stages) & 1u);
        const uint8_t* row = ring + (size_t)s * row_bytes;
#pragma unroll
        for (int k = 0; k < K4; ++k) {
            const int v = lane + 32 * k;
            cur[k] = (EXACT || v < nv4) ? *reinterpret_cast<const uint2*>(row + 8 * v) : make_uint2(0u, 0u);
        }
        // ---- norm: 4 accumulators per lane, sequential over k (ATen Reduce.cuh, input_vec_size 4)
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int k = 0; k < K4; ++k) {
            fma_sq_bf16x2(a0, a1, cur[k].x);
            fma_sq_bf16x2(a2, a3, cur[k].y);
        }
        float ss = ((a0 + a1) + a2) + a3;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) ss += __shfl_down_sync(0xffffffffu, ss, off);
        ss = __shfl_sync(0xffffffffu, ss, 0);
        // the ring slot is free again (all lanes hold their copy in registers): refill it
        __syncwarp();
        if (lane == 0 && prod.valid()) { issue(prod, s); prod.advance(); }

        float nrm = round_bf16(__fsqrt_rn(ss));
        nrm = fmaxf(nrm, eps);
        if (AUX) {
            if (lane == 0) aux.nrm[(size_t)cons.f * aux.si + (size_t)cons.p * aux.sp] = nrm;
        }
        const float rcp = __frcp_rn(nrm);
#pragma unroll
        for (int k = 0; k < K4; ++k) {
            cur[k].x = scale_bf16x2_rn(cur[k].x, rcp);
            cur[k].y = scale_bf16x2_rn(cur[k].y, rcp);
        }
        if (cons.f != cons.fbeg) {
            // ---- sum of rounded products in the 8-element-vector order (Reduce.cuh, input_vec_size 8):
            // 8-vector l'+32k' = 4-vectors (2l'+h)+64k'; for l'<16 they sit in lanes 2l'+h at even k,
            // for l'>=16 in lanes 2(l'-16)+h at odd k.
            float e0 = 0.f, e1 = 0.f, e2 = 0.f, e3 = 0.f, o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f;
#pragma unroll
            for (int k = 0; k < K4; ++k) {
                const uint32_t p01 = mul_bf16x2_rn(prev[k].x, cur[k].x);
                const uint32_t p23 = mul_bf16x2_rn(prev[k].y, cur[k].y);
                if ((k & 1) == 0) {
                    add_bf16x2(e0, e1, p01);
                    add_bf16x2(e2, e3, p23);
                } else {
                    add_bf16x2(o0, o1, p01);
                    add_bf16x2(o2, o3, p23);
                }
            }
            const float se = ((e0 + e1) + e2) + e3;          // accumulators 0..3 of 8-lane l' (even lanes)
            const float so = ((o0 + o1) + o2) + o3;
            const float te = __shfl_up_sync(0xffffffffu, se, 1);
            const float to = __shfl_up_sync(0xffffffffu, so, 1);
            const float ve = (((te + e0) + e1) + e2) + e3;   // odd lanes: full 8-accumulator fold
            const float vo = (((to + o0) + o1) + o2) + o3;
            float v = ve + vo;                               // shfl-down offset 16 in 8-lane space
            v += __shfl_down_sync(0xffffffffu, v, 16);       // offset 8
            v += __shfl_down_sync(0xffffffffu, v, 8);        // offset 4
            v += __shfl_down_sync(0xffffffffu, v, 4);        // offset 2
            v += __shfl_down_sync(0xffffffffu, v, 2);        // offset 1  -> 8-lane 0 == physical lane 1
            if (lane == 1) {
                if (AUX) aux.sim[(size_t)(cons.f - 1) * aux.si + (size_t)cons.p * aux.sp] = round_bf16(v);   // MA-LLM state
                else dis[(size_t)(cons.f - halo) * N + cons.p] = 1.0f - round_bf16(v);
            }
        } else if (!AUX && cons.f == 0 && !halo) {
            if (lane == 0) dis[cons.p] = 1.0f;
        }
        ++consumed;
        cons.advance();
    };
    uint2 ra[K4], rb[K4];                                    // normalised rows, bf16x2 packed (ping-pong)
    while (cons.valid()) {
        process_row(ra, rb);
        if (!cons.valid()) break;
        process_row(rb, ra);
    }
}

__global__ void fill_f32_kernel(float* p, int n, float v) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

template <int K4, bool AUX = false>
static int launch_dis(const void* x, int T, int N, int C, int halo, float* dis, cudaStream_t st, DisAux aux = DisAux{nullptr, nullptr, 0, 0}) {
    int dev = 0, sms = 0, smem_max = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    const size_t row_bytes = (size_t)C * 2;
    const int ctas_per_sm = (K4 <= 16) ? 2 : 1;
    int active = kDisWarps;
    int stages = (int)(((size_t)smem_max / ctas_per_sm - 2048) / (active * row_bytes));
    while (stages < 2 && active > 2) {                         // very long rows: fewer streaming warps, deeper rings
        active >>= 1;
        stages = (int)(((size_t)smem_max / ctas_per_sm - 2048) / (active * row_bytes));
    }
    if (stages > 8) stages = 8;
    if (stages < 2) return RTK_E_UNSUPPORTED;
    const size_t smem = (size_t)active * stages * row_bytes + (size_t)kDisWarps * stages * 8;
    // run length: long enough that the halo re-read is small, short enough to give every warp >= 4 items
    const long long frames = T - 1;
    const long long warps = (long long)sms * active * ctas_per_sm;
    long long R = (frames * N) / (warps * 4);
    if (R > 32) R = 32;
    if (R < 4) R = 4;
    if (R > frames) R = frames;
    const long long runs = (frames + R - 1) / R;
    const long long n_items = runs * N;
    long long grid = (n_items + active - 1) / active;
    if (grid > (long long)sms * ctas_per_sm) grid = (long long)sms * ctas_per_sm;
    auto kern = (!AUX && C == K4 * 128) ? dpselect_dis_kernel<K4, AUX, !AUX> : dpselect_dis_kernel<K4, AUX, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    kern<<<(unsigned)grid, kDisThreads, smem, st>>>((const __nv_bfloat16*)x, dis, T, N, C, (int)R, (int)n_items,
                                                     stages, halo, aux, active);
    RTK_CHECK_LAUNCH();
    return 0;
}

// ============================================================================================== A2: select
constexpr int kSelWarps = 8;

// one warp: indices of the t largest keys of `keys[0..T)` (radix-ordered uint32) in ascending index order;
// ties at the threshold go to the lowest indices (ATen sbtopk/mbtopk gather order).
template <typename Emit>
__device__ __forceinline__ void warp_select_top(const uint32_t* keys, int T, int t, int lane, Emit emit) {
    uint32_t prefix = 0;
    for (int bit = 31; bit >= 0; --bit) {
        const uint32_t cand = prefix | (1u << bit);
        int cnt = 0;
        for (int i = lane; i < T; i += 32) cnt += (keys[i] >= cand);
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (cnt >= t) prefix = cand;
    }
    int gt = 0;
    for (int i = lane; i < T; i += 32) gt += (keys[i] > prefix);
    gt = __reduce_add_sync(0xffffffffu, gt);
    const int need = t - gt;                                  // equal keys to take, lowest index first
    int kept = 0, eqs = 0;
    const uint32_t lt = (1u << lane) - 1u;
    for (int base = 0; base < T; base += 32) {
        const int i = base + lane;
        const uint32_t key = (i < T) ? keys[i] : 0u;
        const bool is_eq = (i < T) && key == prefix;
        const uint32_t beq = __ballot_sync(0xffffffffu, is_eq);
        const bool keep = (i < T) && (key > prefix || (is_eq && eqs + __popc(beq & lt) < need));
        const uint32_t bk = __ballot_sync(0xffffffffu, keep);
        if (keep) emit(kept + __popc(bk & lt), i);
        kept += __popc(bk);
        eqs += __popc(beq);
    }
}

__device__ __forceinline__ bool is_peak(const float* d, int i, int T) {
    // ATen's max_pool1d_with_indices(window 3, pad 1) window loop, literally: the argmax starts at the window's first
    // valid position with max -inf, and v is taken when v > max || isnan(v).  On finite values that keeps the first
    // maximum (strict on the left, >= on the right); in a run of NaNs it keeps the LAST NaN of the window.
    int arg = max(i - 1, 0);
    float mx = -INFINITY;
#pragma unroll
    for (int u = -1; u <= 1; ++u) {
        const int j = i + u;
        if (j < 0 || j >= T) continue;
        const float v = d[j];
        if (v > mx || v != v) {
            mx = v;
            arg = j;
        }
    }
    return arg == i;
}

// sync == 0: a CTA of W warps (W = blockDim.x / 32, a power of two <= 8) handles W consecutive patch columns, one warp
// each; W is chosen by the host so that the grid covers the machine (few patches per CTA when N is small).
__global__ void __launch_bounds__(kSelWarps * kWarp)
dpselect_select_patch_kernel(const float* __restrict__ dis, int T, int N, int t, int32_t* __restrict__ idx,
                             uint8_t* __restrict__ mask) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int W = blockDim.x >> 5;
    float* sd = reinterpret_cast<float*>(smem);               // [W][T] raw distances, then radix keys in place
    uint8_t* spk = smem + (size_t)W * T * 4;                  // [W][T] peak flags
    const int p0 = blockIdx.x * W;
    const int np = min(W, N - p0);
    {   // thread (tt0, j) walks frames tt0, tt0 + 32, ...; 8 independent loads in flight per thread
        const int j = threadIdx.x & (W - 1), tt0 = threadIdx.x / W;
        constexpr int kStep = kWarp;                                  // frames covered per sweep of the block
        if (j < np) {
            const float* src = dis + p0 + j;
            float* dst = sd + j * T;
            int tt = tt0;
            for (; tt + 7 * kStep < T; tt += 8 * kStep) {
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = __ldg(src + (size_t)(tt + u * kStep) * N);
#pragma unroll
                for (int u = 0; u < 8; ++u) dst[tt + u * kStep] = v[u];
            }
            for (; tt < T; tt += kStep) dst[tt] = __ldg(src + (size_t)tt * N);
        }
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp >= np) return;
    float* d = sd + warp * T;
    uint8_t* pk = spk + warp * T;
    for (int i = lane; i < T; i += 32) pk[i] = is_peak(d, i, T);
    __syncwarp();
    uint32_t* keys = reinterpret_cast<uint32_t*>(d);
    for (int i = lane; i < T; i += 32) {
        const float v = pk[i] ? d[i] + 2.0f : d[i];
        keys[i] = f32_to_ordered(v);
    }
    __syncwarp();
    const int p = p0 + warp;
    warp_select_top(keys, T, t, lane, [&](int slot, int i) {
        idx[(size_t)slot * N + p] = i;
        mask[(size_t)slot * N + p] = pk[i];
    });
}

// fp32 sum of one contiguous row in the order ATen's CUDA reduce kernel uses for `dis.mean(1)` (Reduce.cuh):
//  n >= 128: "vectorize along input" - an unaligned head (lanes shift..3 take one element each), then lane l owns
//            the aligned float4 vectors l, l+32, ... with one accumulator per vector element, then a scalar tail
//            folded into accumulator 0;
//  n <  128: block width bw = min(last_pow2(n), 32); lane l owns elements l, l+bw, ... dealt round-robin to four
//            accumulators;
// accumulators are folded ((a0+a1)+a2)+a3 and lanes with a shfl-down tree.  Result valid in lane 0.
__device__ __forceinline__ float aten_row_sum_f32(const float* __restrict__ row, int n, int lane) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int width = 32;
    if (n >= 128) {
        const float* data = row;
        int end = n;
        const int shift = (int)(((uintptr_t)row & 15u) >> 2);
        if (shift > 0) {
            data -= shift;
            end += shift;
            if (lane >= shift && lane < 4) a0 = a0 + data[lane];
            end -= 4;
            data += 4;
        }
        for (int idx = lane; idx * 4 + 3 < end; idx += 32) {
            const float4 q = *reinterpret_cast<const float4*>(data + 4 * idx);
            a0 += q.x; a1 += q.y; a2 += q.z; a3 += q.w;
        }
        const int tail = end - end % 4 + lane;
        if (tail < end) a0 += data[tail];
    } else {
        width = 1;
        while (width * 2 <= n && width < 32) width *= 2;
        if (lane < width) {
            int idx = lane;
            while (idx + 3 * width < n) {
                a0 += row[idx]; a1 += row[idx + width]; a2 += row[idx + 2 * width]; a3 += row[idx + 3 * width];
                idx += 4 * width;
            }
            if (idx < n) { a0 += row[idx]; idx += width; }
            if (idx < n) { a1 += row[idx]; idx += width; }
            if (idx < n) { a2 += row[idx]; idx += width; }
            if (idx < n) { a3 += row[idx]; }
        }
    }
    float s = ((a0 + a1) + a2) + a3;
    for (int off = width >> 1; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
    return s;
}

// sync == 1: per-frame mean over patches (ATen mean: fp32 sum in Reduce.cuh order with 4-element vectors,
// times fp32(1/N)), then one warp selects frames; the mask row of each kept frame is replicated N times.
constexpr int kSyncWarps = 32;    // one CTA; 32 row means in flight instead of 8 (the means are a chain of DRAM round trips)
__global__ void __launch_bounds__(kSyncWarps * kWarp)
dpselect_select_sync_kernel(const float* __restrict__ dis, int T, int N, int t, int32_t* __restrict__ idx,
                            uint8_t* __restrict__ mask) {
    extern __shared__ __align__(128) uint8_t smem[];
    float* d = reinterpret_cast<float*>(smem);                // [T]
    uint8_t* pk = smem + (size_t)T * 4;                       // [T]
    int32_t* sel = reinterpret_cast<int32_t*>(smem + (size_t)T * 4 + (((size_t)T + 15) & ~(size_t)15));  // [t]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float rcpN = 1.0f / (float)N;
    for (int tt = warp; tt < T; tt += kSyncWarps) {
        const float s = aten_row_sum_f32(dis + (size_t)tt * N, N, lane);
        if (lane == 0) d[tt] = s * rcpN;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < T; i += blockDim.x) pk[i] = is_peak(d, i, T);
    __syncthreads();
    uint32_t* keys = reinterpret_cast<uint32_t*>(d);
    for (int i = threadIdx.x; i < T; i += blockDim.x) {
        const float v = pk[i] ? d[i] + 2.0f : d[i];
        keys[i] = f32_to_ordered(v);
    }
    __syncthreads();
    if (warp == 0) {
        warp_select_top(keys, T, t, lane, [&](int slot, int i) {
            sel[slot] = i;
            idx[slot] = i;
        });
    }
    __syncthreads();
    // mask row of kept frame j = its peak flag, N times: 16-byte stores where the row allows it
    for (int j = warp; j < t; j += kSyncWarps) {
        const uint8_t f = pk[sel[j]];
        uint8_t* row = mask + (size_t)j * N;
        const int head = min(N, (int)((16 - ((uintptr_t)row & 15)) & 15));
        const int body = (N - head) >> 4;
        const uint4 w = make_uint4(f * 0x01010101u, f * 0x01010101u, f * 0x01010101u, f * 0x01010101u);
        for (int i = lane; i < head; i += 32) row[i] = f;
        for (int i = lane; i < body; i += 32) reinterpret_cast<uint4*>(row + head)[i] = w;
        for (int i = head + body * 16 + lane; i < N; i += 32) row[i] = f;
    }
}

// ============================================================================================== A3: gather
// out[j, p, :] = x[idx[...], p, :]; one warp per output row, 16-byte vectors, 8 loads in flight per lane.
// Frame-range split (SURVEY.md 8e): x holds frames [frame_first, ...) of the video and only output rows whose source frame
// lies in [t0, t1) are written (the others belong to other ranks); the single-GPU call passes 0, 0, INT_MAX.
__global__ void __launch_bounds__(256)
dpselect_gather_kernel(const uint4* __restrict__ x, const int32_t* __restrict__ idx, uint4* __restrict__ out,
                       int N, int nvec, long long rows, int sync, int frame_first, int t0, int t1) {
    const int lane = threadIdx.x & 31;
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long GW = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = gw; r < rows; r += GW) {
        const long long j = r / N;
        const int p = (int)(r - j * N);
        const int src_t = sync ? idx[j] : idx[r];
        if (src_t < t0 || src_t >= t1) continue;
        const uint4* src = x + ((size_t)(src_t - frame_first) * N + p) * (size_t)nvec;
        uint4* dst = out + (size_t)r * nvec;
        int v = lane;
        for (; v + 7 * 32 < nvec; v += 8 * 32) {
            uint4 b[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) b[u] = __ldg(src + v + 32 * u);
#pragma unroll
            for (int u = 0; u < 8; ++u) dst[v + 32 * u] = b[u];
        }
        for (; v < nvec; v += 32) dst[v] = __ldg(src + v);
    }
}

// generic row gather: out[i, :] = x[src_row[i], :], rows of nvec 16-byte vectors (frame-range-sharded compaction)
__global__ void __launch_bounds__(256)
gather_rows_kernel(const uint4* __restrict__ x, const long long* __restrict__ src_row, uint4* __restrict__ out, int nvec,
                   long long rows) {
    const int lane = threadIdx.x & 31;
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long GW = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = gw; r < rows; r += GW) {
        const uint4* src = x + (size_t)src_row[r] * nvec;
        uint4* dst = out + (size_t)r * nvec;
        int v = lane;
        for (; v + 7 * 32 < nvec; v += 8 * 32) {
            uint4 b[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) b[u] = __ldg(src + v + 32 * u);
#pragma unroll
            for (int u = 0; u < 8; ++u) dst[v + 32 * u] = b[u];
        }
        for (; v < nvec; v += 32) dst[v] = __ldg(src + v);
    }
}

// adjacent-frame similarities (bf16-valued) and clamped row norms into strided state arrays: the first pass of the
// MA-LLM compressors (mallm.cu) on the streaming kernel above
int dpselect_sim_nrm(const void* x, int64_t T, int64_t N, int64_t C, DisAux aux, cudaStream_t st) {
    if (T < 2) return RTK_E_BADARG;
    const int k4 = (int)((C / 4 + 31) / 32);
    if (k4 <= 2) return launch_dis<2, true>(x, (int)T, (int)N, (int)C, 0, nullptr, st, aux);
    if (k4 <= 4) return launch_dis<4, true>(x, (int)T, (int)N, (int)C, 0, nullptr, st, aux);
    if (k4 <= 9) return launch_dis<9, true>(x, (int)T, (int)N, (int)C, 0, nullptr, st, aux);
    if (k4 <= 16) return launch_dis<16, true>(x, (int)T, (int)N, (int)C, 0, nullptr, st, aux);
    if (k4 <= 28) return launch_dis<28, true>(x, (int)T, (int)N, (int)C, 0, nullptr, st, aux);
    if (k4 <= 32) return launch_dis<32, true>(x, (int)T, (int)N, (int)C, 0, nullptr, st, aux);
    if (k4 <= 48) return launch_dis<48, true>(x, (int)T, (int)N, (int)C, 0, nullptr, st, aux);
    return launch_dis<64, true>(x, (int)T, (int)N, (int)C, 0, nullptr, st, aux);
}

}  // namespace rtk

// =================================================================================================== C ABI
using namespace rtk;

extern "C" int rtk_dpselect_dis(const void* x, int64_t T, int64_t N, int64_t C, int halo, float* dis, void* stream) {
    RTK_NVTX("rtk_dpselect_dis");
    if (!x || !dis || T < 1 || N < 1) return RTK_E_BADARG;
    if (C % 8 != 0 || C < 256 || C > 8192) return RTK_E_UNSUPPORTED;
    if (((uintptr_t)x & 15u) != 0) return RTK_E_ALIGN;
    if (T > (1 << 20) || N > (1 << 20) || T * N > (1ll << 31) - 1) return RTK_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (T == 1) {
        if (halo) return 0;
        fill_f32_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(dis, (int)N, 1.0f);
        RTK_CHECK_LAUNCH();
        return 0;
    }
    const int k4 = (int)((C / 4 + 31) / 32);
    if (k4 <= 2) return launch_dis<2>(x, (int)T, (int)N, (int)C, halo, dis, st);
    if (k4 <= 4) return launch_dis<4>(x, (int)T, (int)N, (int)C, halo, dis, st);
    if (k4 <= 9) return launch_dis<9>(x, (int)T, (int)N, (int)C, halo, dis, st);
    if (k4 <= 16) return launch_dis<16>(x, (int)T, (int)N, (int)C, halo, dis, st);
    if (k4 <= 28) return launch_dis<28>(x, (int)T, (int)N, (int)C, halo, dis, st);
    if (k4 <= 32) return launch_dis<32>(x, (int)T, (int)N, (int)C, halo, dis, st);
    if (k4 <= 48) return launch_dis<48>(x, (int)T, (int)N, (int)C, halo, dis, st);
    return launch_dis<64>(x, (int)T, (int)N, (int)C, halo, dis, st);
}

extern "C" int rtk_dpselect_select(const float* dis, int64_t T, int64_t N, int64_t t, int sync, int32_t* idx,
                                   uint8_t* mask, void* stream) {
    RTK_NVTX("rtk_dpselect_select");
    if (!dis || !idx || !mask || T < 1 || N < 1 || t < 1 || t > T) return RTK_E_BADARG;
    if (T > 8192) return RTK_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (sync) {
        if (((uintptr_t)dis & 3u) != 0) return RTK_E_ALIGN;
        const size_t smem = (size_t)T * 4 + (((size_t)T + 15) & ~(size_t)15) + (size_t)t * 4;
        cudaError_t e = cudaFuncSetAttribute(dpselect_select_sync_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)smem);
        if (e != cudaSuccess) return (int)e;
        dpselect_select_sync_kernel<<<1, kSyncWarps * kWarp, smem, st>>>(dis, (int)T, (int)N, (int)t, idx, mask);
    } else {
        int dev = 0, smem_max = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        int W = kSelWarps;                                      // patches per CTA: fewer when that still leaves >= ~2 CTAs per SM
        while (W > 1 && (N + W - 1) / W < 296) W >>= 1;
        // and fewer when W columns of T distances + peak flags do not fit (8 columns stop fitting at T = 5812 on a B200;
        // one warp per column, so W does not change the result)
        while (W > 1 && (size_t)W * T * 5 > (size_t)smem_max) W >>= 1;
        const size_t smem = (size_t)W * T * 5;
        cudaError_t e = cudaFuncSetAttribute(dpselect_select_patch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)smem);
        if (e != cudaSuccess) return (int)e;
        const unsigned grid = (unsigned)((N + W - 1) / W);
        dpselect_select_patch_kernel<<<grid, W * kWarp, smem, st>>>(dis, (int)T, (int)N, (int)t, idx, mask);
    }
    RTK_CHECK_LAUNCH();
    return 0;
}

extern "C" int rtk_dpselect_gather(const void* x, int64_t T, int64_t N, int64_t C, const int32_t* idx, int64_t t,
                                   int sync, void* out, void* stream) {
    RTK_NVTX("rtk_dpselect_gather");
    if (!x || !idx || !out || T < 1 || N < 1 || C < 1 || t < 1) return RTK_E_BADARG;
    if (C % 8 != 0) return RTK_E_UNSUPPORTED;
    if ((((uintptr_t)x | (uintptr_t)out) & 15u) != 0) return RTK_E_ALIGN;
    if (t > T) return RTK_E_BADARG;
    // (t == T, the shipped compression_ratio 1.0, is the identity: the same kernel copies it - no copy-engine shortcut,
    //  so that the operator's bandwidth figure is this library's own)
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long rows = (long long)t * N;
    long long grid = (rows + 7) / 8;
    if (grid > (long long)sms * 8) grid = (long long)sms * 8;
    dpselect_gather_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(
        (const uint4*)x, idx, (uint4*)out, (int)N, (int)(C / 8), rows, sync, 0, 0, INT_MAX);
    RTK_CHECK_LAUNCH();
    return 0;
}

extern "C" int rtk_dpselect_gather_owned(const void* x_local, int64_t frames_local, int64_t frame_first, int64_t t0, int64_t t1,
                                         int64_t N, int64_t C, const int32_t* idx, int64_t t, int sync, void* out, void* stream) {
    RTK_NVTX("rtk_dpselect_gather_owned");
    if (!x_local || !idx || !out || frames_local < 1 || N < 1 || C < 1 || t < 1) return RTK_E_BADARG;
    if (t0 < frame_first || t1 > frame_first + frames_local || t0 > t1) return RTK_E_BADARG;
    if (C % 8 != 0) return RTK_E_UNSUPPORTED;
    if ((((uintptr_t)x_local | (uintptr_t)out) & 15u) != 0) return RTK_E_ALIGN;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long rows = (long long)t * N;
    long long grid = (rows + 7) / 8;
    if (grid > (long long)sms * 8) grid = (long long)sms * 8;
    dpselect_gather_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(
        (const uint4*)x_local, idx, (uint4*)out, (int)N, (int)(C / 8), rows, sync, (int)frame_first, (int)t0, (int)t1);
    RTK_CHECK_LAUNCH();
    return 0;
}

// the whole operator in one call: one crossing of the FFI, three back-to-back launches
extern "C" int rtk_dpselect_keyframe(const void* x, int64_t T, int64_t N, int64_t C, int64_t t, int sync, float* dis,
                                     int32_t* idx, uint8_t* mask, void* out, void* stream) {
    RTK_NVTX("rtk_dpselect_keyframe");
    int rc = rtk_dpselect_dis(x, T, N, C, 0, dis, stream);
    if (rc) return rc;
    rc = rtk_dpselect_select(dis, T, N, t, sync, idx, mask, stream);
    if (rc) return rc;
    return rtk_dpselect_gather(x, T, N, C, idx, t, sync, out, stream);
}

extern "C" int rtk_gather_rows(const void* x, int64_t row_bytes, const int64_t* src_row, int64_t rows, void* out,
                               void* stream) {
    RTK_NVTX("rtk_gather_rows");
    if (!x || !src_row || !out || rows < 0 || row_bytes < 16) return RTK_E_BADARG;
    if (row_bytes % 16 != 0) return RTK_E_UNSUPPORTED;
    if ((((uintptr_t)x | (uintptr_t)out) & 15u) != 0) return RTK_E_ALIGN;
    if (rows == 0) return 0;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long grid = (rows + 7) / 8;
    if (grid > (long long)sms * 8) grid = (long long)sms * 8;
    gather_rows_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>((const uint4*)x, (const long long*)src_row,
                                                                        (uint4*)out, (int)(row_bytes / 16), rows);
    RTK_CHECK_LAUNCH();
    return 0;
}
