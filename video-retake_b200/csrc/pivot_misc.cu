// PivotKV side kernels (sm_100a): rotary (un)rotation, KV-head mean + top-k selection, KV / position compaction.
// Replaces retake/longvideo_cache.py:248-259 (B0), :270-277 (B2), :278-306 (B3).
#include <climits>

#include <stdlib.h>

#include "rtk_common.cuh"

namespace rtk {

// ======================================================================================== B0: rotary
struct RopeParams {
    int heads, L, D, n_pos, forward;
    long long stride_h, stride_l, out_stride_h, out_stride_l;
    // optional second tensor handled by the same launch (k next to q): heads [heads, heads + heads2)
    int heads2;
    const __nv_bfloat16* x2;
    __nv_bfloat16* out2;
    long long stride_h2, stride_l2, out_stride_h2, out_stride_l2;
    int bound[6];            // exclusive channel boundaries of the six mrope blocks (sections * 2)
    float inv_scale2;
};

// RopeParams::bound from the mrope sections (all zero unless n_pos == 3); false when 3-D sections do not cover D
static bool mrope_bounds(int n_pos, const int32_t* sec, int64_t D, int bound[6]) {
    int acc = 0;
    for (int i = 0; i < 6; ++i) {
        acc += n_pos == 3 ? sec[i % 3] : 0;
        bound[i] = acc;
    }
    return n_pos != 3 || acc == D;
}

__device__ __forceinline__ int rope_pos_row(const RopeParams& p, int c) {
    if (p.n_pos == 1) return 0;
    int i = 0;
    while (i < 5 && c >= p.bound[i]) ++i;
    return i % 3;
}

// cos/sin tables of one chunk straight from the rotary module's inv_freq: what HF's rotary forward computes
// (freqs = inv_freq * pos in fp32, emb = cat(freqs, freqs), cos(emb) * attention_scaling -> bf16), already
// reduced to the one position row each channel uses under mrope.  Replaces ~12 small torch launches per call.
__global__ void __launch_bounds__(256)
pivot_rope_table_kernel(const long long* __restrict__ pos, const float* __restrict__ inv_freq, RopeParams p, float scaling,
                        __nv_bfloat16* __restrict__ cos_t, __nv_bfloat16* __restrict__ sin_t) {
    pdl_enter();
    const int half = p.D >> 1;
    const long long total = (long long)p.L * p.D;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % p.D);
        const int l = (int)(i / p.D);
        const long long pv = pos[(size_t)rope_pos_row(p, c) * p.L + l];
        const float ang = inv_freq[c < half ? c : c - half] * (float)pv;
        cos_t[i] = __float2bfloat16_rn(cosf(ang) * scaling);
        sin_t[i] = __float2bfloat16_rn(sinf(ang) * scaling);
    }
}

// channel c of the lower half (xa, tables cosa/sina) and its partner c + D/2 (xb, cosb/sinb), every product and sum
// rounded to bf16 like the reference's op-by-op bf16 expression (longvideo_cache.py:36-83)
__device__ __forceinline__ void rope_rotate_pair(float xa, float xb, float cosa, float sina, float cosb, float sinb, int forward,
                                                 float inv_scale2, __nv_bfloat16& oa, __nv_bfloat16& ob) {
    // rotate_half: lower half pairs with -x[c + D/2], upper half with +x[c - D/2]
    const float ta = round_bf16(xa * cosa), ra = round_bf16(-xb * sina);
    const float tb = round_bf16(xb * cosb), rb = round_bf16(xa * sinb);
    float ya, yb;
    if (forward) {
        ya = ta + ra;
        yb = tb + rb;
    } else {
        ya = round_bf16(ta - ra) * inv_scale2;
        yb = round_bf16(tb - rb) * inv_scale2;
    }
    oa = __float2bfloat16_rn(ya);
    ob = __float2bfloat16_rn(yb);
}

// cos/sin of channel c at the positions pv[0..n_pos) of one token, as the HF rotary module computes them
__device__ __forceinline__ void rope_table_entry(const RopeParams& p, const float* __restrict__ inv_freq, const long long* pv,
                                                 int c, float scaling, float& co, float& si) {
    const int half = p.D >> 1;
    const float ang = inv_freq[c < half ? c : c - half] * (float)pv[rope_pos_row(p, c)];
    co = __bfloat162float(__float2bfloat16_rn(cosf(ang) * scaling));
    si = __bfloat162float(__float2bfloat16_rn(sinf(ang) * scaling));
}

// Reverse rotation of q and k with the tables computed in place (fast path: the rotary module has a static inv_freq):
// one CTA per token, D threads build the token's cos/sin row in shared memory, then every thread rotates one
// (head, 8+8 channel) slice of q or k.  Replaces pivot_rope_table_kernel + pivot_rope_kernel of the slow path.
#ifndef RTK_UNROPE_TOK
#define RTK_UNROPE_TOK 2     // A/B under ncu, 28 layers x 4096 tokens: 1 -> 597 us, 2 -> 538 us, 4 -> 692 us (100 registers), 8 -> 653 us
#endif
constexpr int kUnropeTok = RTK_UNROPE_TOK;      // tokens a CTA un-rotates per step: their rows are all in flight before the first is used

// packed bf16 arithmetic with ONE rounding per operation.  The reference's chain rounds every product and every
// difference to bf16 after computing it in fp32; for bf16 operands (p = 8 bits) the fp32 intermediate (24 >= 2p + 2 bits)
// makes that double rounding innocuous, so mul / add / sub.rn.bf16x2 return the same bits with a quarter of the instructions.
__device__ __forceinline__ uint32_t sub_bf16x2_rn(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("sub.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ uint32_t add_bf16x2_rn(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("add.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
// reverse rotation of two channel pairs: xa = channels (c, c+1) of the lower half, xb = their partners (c + D/2, ...);
// cos / sin of the lower-half channels (the upper half uses the same values, see unrope_qk_body)
__device__ __forceinline__ void unrotate_bf16x2(uint32_t xa, uint32_t xb, uint32_t cs, uint32_t sn, bool scale, float inv_scale2,
                                                uint32_t& oa, uint32_t& ob) {
    const uint32_t ta = mul_bf16x2_rn(xa, cs), ra = mul_bf16x2_rn(xb ^ 0x80008000u, sn);     // rotate_half: -x[c + D/2]
    const uint32_t tb = mul_bf16x2_rn(xb, cs), rb = mul_bf16x2_rn(xa, sn);
    oa = sub_bf16x2_rn(ta, ra);
    ob = sub_bf16x2_rn(tb, rb);
    if (scale) {
        oa = scale_bf16x2_rn(oa, inv_scale2);
        ob = scale_bf16x2_rn(ob, inv_scale2);
    }
}

__device__ __forceinline__ void unrope_qk_body(const __nv_bfloat16* __restrict__ x, const long long* __restrict__ pos,
                                               const float* __restrict__ inv_freq, float scaling,
                                               __nv_bfloat16* __restrict__ out, const RopeParams& p) {
    // cos / sin rows of the step's tokens, LOWER half of the channels only: emb = cat(freqs, freqs) and the mrope blocks
    // i and i + 3 read the same position row (sections sum to D / 2), so channel c + D/2 has the tables of channel c
    __shared__ __align__(16) __nv_bfloat16 s_cos[kUnropeTok][128], s_sin[kUnropeTok][128];
    const int half = p.D >> 1;
    const int vec_per_row = half >> 3;
    const int ntask = (p.heads + p.heads2) * vec_per_row;
    const int tid = threadIdx.x;
    const bool scale = p.inv_scale2 != 1.0f;
    // a thread's first task (at the 7B shape - 32 heads x 8 vectors - its only one): same (head, vector) for every token
    const int v0 = tid % vec_per_row, h0 = tid / vec_per_row;
    const bool second0 = h0 >= p.heads;
    const long long src_h0 = second0 ? (long long)(h0 - p.heads) * p.stride_h2 : (long long)h0 * p.stride_h;
    const long long src_l0 = second0 ? p.stride_l2 : p.stride_l;
    const __nv_bfloat16* src0 = (second0 ? p.x2 : x) + src_h0 + v0 * 8;
    for (int l0 = blockIdx.x * kUnropeTok; l0 < p.L; l0 += gridDim.x * kUnropeTok) {
        const int nl = min(kUnropeTok, p.L - l0);
        // every row of the step is requested before the tables are built, so that the trigonometry hides the latency
        uint4 lo4[kUnropeTok], hi4[kUnropeTok];
        if (tid < ntask) {
#pragma unroll
            for (int t = 0; t < kUnropeTok; ++t) {
                if (t < nl) {
                    lo4[t] = *reinterpret_cast<const uint4*>(src0 + (l0 + t) * src_l0);
                    hi4[t] = *reinterpret_cast<const uint4*>(src0 + (l0 + t) * src_l0 + half);
                }
            }
        }
        for (int e = tid; e < nl * half; e += blockDim.x) {
            const int t = e / half, c = e - t * half;
            long long pv[3] = {0, 0, 0};
            for (int r = 0; r < p.n_pos; ++r) pv[r] = pos[(size_t)r * p.L + l0 + t];
            float co, si;
            rope_table_entry(p, inv_freq, pv, c, scaling, co, si);
            s_cos[t][c] = __float2bfloat16_rn(co);          // exact: the entries are bf16 values already
            s_sin[t][c] = __float2bfloat16_rn(si);
        }
        __syncthreads();
#pragma unroll
        for (int t = 0; t < kUnropeTok; ++t) {
            if (t >= nl) break;
            const int l = l0 + t;
            for (int task = tid; task < ntask; task += blockDim.x) {
                const int v = task % vec_per_row, h = task / vec_per_row;
                const int c0 = v * 8;
                const bool second = h >= p.heads;
                const __nv_bfloat16* src = second ? p.x2 + (h - p.heads) * p.stride_h2 + l * p.stride_l2 : x + h * p.stride_h + l * p.stride_l;
                __nv_bfloat16* dst = second ? p.out2 + (h - p.heads) * p.out_stride_h2 + l * p.out_stride_l2
                                            : out + h * p.out_stride_h + l * p.out_stride_l;
                uint4 a4 = lo4[t], b4 = hi4[t];
                if (task != tid) {
                    a4 = *reinterpret_cast<const uint4*>(src + c0);
                    b4 = *reinterpret_cast<const uint4*>(src + c0 + half);
                }
                const uint4 cs = *reinterpret_cast<const uint4*>(&s_cos[t][c0]);
                const uint4 sn = *reinterpret_cast<const uint4*>(&s_sin[t][c0]);
                uint4 ol4, oh4;
                unrotate_bf16x2(a4.x, b4.x, cs.x, sn.x, scale, p.inv_scale2, ol4.x, oh4.x);
                unrotate_bf16x2(a4.y, b4.y, cs.y, sn.y, scale, p.inv_scale2, ol4.y, oh4.y);
                unrotate_bf16x2(a4.z, b4.z, cs.z, sn.z, scale, p.inv_scale2, ol4.z, oh4.z);
                unrotate_bf16x2(a4.w, b4.w, cs.w, sn.w, scale, p.inv_scale2, ol4.w, oh4.w);
                *reinterpret_cast<uint4*>(dst + c0) = ol4;
                *reinterpret_cast<uint4*>(dst + c0 + half) = oh4;
            }
        }
        __syncthreads();
    }
}

// Per-layer tables of an update (rtk_pivot_update_batch; rtk_pivot_update is a batch of one): every layer of the chunk
// brings its own tensors, the shapes are shared.  Passed as ONE __grid_constant__ kernel parameter (4.9 KB).
struct BatchLayers {
    const __nv_bfloat16* q[kMaxBatchLayers];         // caller's views (un-rotation input)
    const __nv_bfloat16* k[kMaxBatchLayers];         // K the compaction reads (the un-rotated copy when re-forging)
    const __nv_bfloat16* k_in[kMaxBatchLayers];      // caller's K view (un-rotation input)
    const __nv_bfloat16* v[kMaxBatchLayers];
    __nv_bfloat16* qu[kMaxBatchLayers];              // un-rotated copies [H, L, D] / [KVH, L, D] in the workspace
    __nv_bfloat16* ku[kMaxBatchLayers];
    const long long* pos[kMaxBatchLayers];
    const uint8_t* keymask[kMaxBatchLayers];
    __nv_bfloat16* k_out[kMaxBatchLayers];
    __nv_bfloat16* v_out[kMaxBatchLayers];
    long long* pos_out[kMaxBatchLayers];
    int32_t* keep_idx[kMaxBatchLayers];
    const __nv_bfloat16* head_scores[kMaxBatchLayers];
    long long q_stride_h[kMaxBatchLayers], q_stride_l[kMaxBatchLayers];
    long long kin_stride_h[kMaxBatchLayers], kin_stride_l[kMaxBatchLayers];
    long long k_stride_h[kMaxBatchLayers], k_stride_l[kMaxBatchLayers];
    long long v_stride_h[kMaxBatchLayers], v_stride_l[kMaxBatchLayers];
    long long out_stride_h[kMaxBatchLayers], pos_out_stride[kMaxBatchLayers];
};

// grid (L, layers): the un-rotation of q and k of every layer of the chunk in one launch
__global__ void __launch_bounds__(256)
pivot_unrope_qk_batch_kernel(const __grid_constant__ BatchLayers t, const float* __restrict__ inv_freq, float scaling, RopeParams p) {
    pdl_enter();
    const int layer = blockIdx.y;
    p.stride_h = t.q_stride_h[layer]; p.stride_l = t.q_stride_l[layer];
    p.x2 = t.k_in[layer]; p.out2 = t.ku[layer];
    p.stride_h2 = t.kin_stride_h[layer]; p.stride_l2 = t.kin_stride_l[layer];
    unrope_qk_body(t.q[layer], t.pos[layer], inv_freq, scaling, t.qu[layer], p);
}

// one thread: 8 channels of the lower half and the 8 partner channels of the upper half of one (head, token)
__global__ void __launch_bounds__(256)
pivot_rope_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ cos_t,
                  const __nv_bfloat16* __restrict__ sin_t, __nv_bfloat16* __restrict__ out, RopeParams p) {
    pdl_enter();
    const int half = p.D >> 1;
    const int vec_per_row = half >> 3;
    const long long total = (long long)(p.heads + p.heads2) * p.L * vec_per_row;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int v = (int)(i % vec_per_row);
        const long long hl = i / vec_per_row;
        const int l = (int)(hl % p.L);
        const int h = (int)(hl / p.L);
        const int c0 = v * 8;
        const bool second = h >= p.heads;
        const __nv_bfloat16* src = second ? p.x2 + (h - p.heads) * p.stride_h2 + l * p.stride_l2 : x + h * p.stride_h + l * p.stride_l;
        __nv_bfloat16* dst = second ? p.out2 + (h - p.heads) * p.out_stride_h2 + l * p.out_stride_l2
                                    : out + h * p.out_stride_h + l * p.out_stride_l;
        uint4 lo4 = *reinterpret_cast<const uint4*>(src + c0);
        uint4 hi4 = *reinterpret_cast<const uint4*>(src + c0 + half);
        const __nv_bfloat16* xl = reinterpret_cast<const __nv_bfloat16*>(&lo4);
        const __nv_bfloat16* xh = reinterpret_cast<const __nv_bfloat16*>(&hi4);
        uint4 ol4, oh4;
        __nv_bfloat16* ol = reinterpret_cast<__nv_bfloat16*>(&ol4);
        __nv_bfloat16* oh = reinterpret_cast<__nv_bfloat16*>(&oh4);
        // cos/sin of the 8 + 8 channels: one 16-byte load each when a vector does not straddle an mrope block
        const int rowa0 = rope_pos_row(p, c0), rowa1 = rope_pos_row(p, c0 + 7);
        const int rowb0 = rope_pos_row(p, c0 + half), rowb1 = rope_pos_row(p, c0 + half + 7);
        uint4 ca4, sa4, cb4, sb4;
        __nv_bfloat16* cav = reinterpret_cast<__nv_bfloat16*>(&ca4);
        __nv_bfloat16* sav = reinterpret_cast<__nv_bfloat16*>(&sa4);
        __nv_bfloat16* cbv = reinterpret_cast<__nv_bfloat16*>(&cb4);
        __nv_bfloat16* sbv = reinterpret_cast<__nv_bfloat16*>(&sb4);
        if (rowa0 == rowa1 && rowb0 == rowb1) {
            const size_t ia = ((size_t)rowa0 * p.L + l) * p.D + c0, ib = ((size_t)rowb0 * p.L + l) * p.D + c0 + half;
            ca4 = __ldg(reinterpret_cast<const uint4*>(cos_t + ia));
            sa4 = __ldg(reinterpret_cast<const uint4*>(sin_t + ia));
            cb4 = __ldg(reinterpret_cast<const uint4*>(cos_t + ib));
            sb4 = __ldg(reinterpret_cast<const uint4*>(sin_t + ib));
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int ca = c0 + e, cb = c0 + e + half;
                const size_t ia = ((size_t)rope_pos_row(p, ca) * p.L + l) * p.D + ca;
                const size_t ib = ((size_t)rope_pos_row(p, cb) * p.L + l) * p.D + cb;
                cav[e] = cos_t[ia]; sav[e] = sin_t[ia]; cbv[e] = cos_t[ib]; sbv[e] = sin_t[ib];
            }
        }
#pragma unroll
        for (int e = 0; e < 8; ++e)
            rope_rotate_pair(__bfloat162float(xl[e]), __bfloat162float(xh[e]), __bfloat162float(cav[e]), __bfloat162float(sav[e]),
                             __bfloat162float(cbv[e]), __bfloat162float(sbv[e]), p.forward, p.inv_scale2, ol[e], oh[e]);
        *reinterpret_cast<uint4*>(dst + c0) = ol4;
        *reinterpret_cast<uint4*>(dst + c0 + half) = oh4;
    }
}

// ================================================================================= key elision (pass 2 of the scoring)
// Key-patch tokens get score 1.0 whatever their column sum is (longvideo_cache.py:272-274 overwrites it before the top-k), so
// the second pass of the scoring - one exp per (query, key) - only has to visit the other keys.  Two small kernels prepare
// that: an exclusive scan of the mask (slot[j] = row of key j among the keys that are NOT key patches, -1 for a key patch;
// n_keys = how many there are) and a gather of those K rows into a compact, token-major copy that pass 2 keeps stationary.
bool key_elision_enabled();

struct KeyElide {
    const uint8_t* keymask[kMaxBatchLayers];     // [L] or nullptr (no key patches: identity)
    int32_t* slot[kMaxBatchLayers];              // [L]
    const __nv_bfloat16* k[kMaxBatchLayers];     // the K rows the scoring uses (un-rotated copy, or the caller's view)
    long long k_stride_h[kMaxBatchLayers], k_stride_l[kMaxBatchLayers];
    __nv_bfloat16* kc[kMaxBatchLayers];          // [n_keys, KVH, D]
    int32_t* n_keys;                             // [layers]
    int L, KVH, D;
};

__global__ void __launch_bounds__(1024)
pivot_keymask_scan_kernel(const __grid_constant__ KeyElide e) {
    pdl_enter();
    __shared__ int wsum[32];
    const int layer = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint8_t* __restrict__ m = e.keymask[layer];
    int32_t* __restrict__ slot = e.slot[layer];
    const int per = (e.L + 1023) / 1024;
    const int beg = min(tid * per, e.L), end = min(beg + per, e.L);
    int cnt = 0;
    for (int i = beg; i < end; ++i) cnt += !(m && m[i]);
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const int w = wsum[lane];
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += n;
        }
        wsum[lane] = winc - w;                               // exclusive over warps
        if (lane == 31) e.n_keys[layer] = winc;
    }
    __syncthreads();
    int base = wsum[warp] + inc - cnt;
    for (int i = beg; i < end; ++i) slot[i] = (m && m[i]) ? -1 : base++;
}

__global__ void __launch_bounds__(256)
pivot_keys_compact_kernel(const __grid_constant__ KeyElide e) {
    pdl_enter();
    const int layer = blockIdx.y;
    const int vpr = e.D >> 3;
    const long long total = (long long)e.L * e.KVH * vpr;
    const int32_t* __restrict__ slot = e.slot[layer];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int v = (int)(i % vpr);
        const long long lh = i / vpr;
        const int h = (int)(lh % e.KVH);
        const int l = (int)(lh / e.KVH);
        const int sl = slot[l];
        if (sl < 0) continue;
        const uint4 w = __ldg(reinterpret_cast<const uint4*>(e.k[layer] + h * e.k_stride_h[layer] + l * e.k_stride_l[layer] + v * 8));
        *reinterpret_cast<uint4*>(e.kc[layer] + ((size_t)sl * e.KVH + h) * e.D + v * 8) = w;
    }
}

// scan + gather for the layers of one launch; fills the elision fields of the scoring batch
static int key_elide_prepare(KeyElide& ke, int n, ScoreBatch& sb, cudaStream_t st) {
    RTK_LAUNCH_PDL(pivot_keymask_scan_kernel, (unsigned)n, 1024, 0, st, ke);
    const long long total = (long long)ke.L * ke.KVH * (ke.D >> 3);
    long long gx = (total + 255) / 256;
    if (gx > 148 * 8) gx = 148 * 8;
    RTK_LAUNCH_PDL(pivot_keys_compact_kernel, dim3((unsigned)gx, (unsigned)n), 256, 0, st, ke);
    for (int i = 0; i < n; ++i) {
        sb.kc[i] = ke.kc[i];
        sb.slot[i] = ke.slot[i];
    }
    sb.n_keys = ke.n_keys;
    return 0;
}

static size_t key_elide_bytes(int64_t KVH, int64_t L, int64_t D) {      // per layer: compact K copy + slots, 256-byte granules
    return (((size_t)KVH * L * D * 2 + 255) & ~(size_t)255) + (((size_t)L * 4 + 255) & ~(size_t)255);
}

// ======================================================================================== B2: select
constexpr int kSelThreads = 1024;

// block-wide: ascending indices of the `keep` largest radix keys in keys[0..L); ties -> lowest index.
__device__ void block_select_top(const uint32_t* keys, int L, int keep, int32_t* out_idx, int* sh /* >= 104 ints */,
                                 int low_bit /* keys are multiples of 2^low_bit */) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (L + kSelThreads - 1) / kSelThreads;
    const int beg = min(tid * per, L), end = min(beg + per, L);
    // bitwise descent for the keep-th largest key: per-warp counts -> shared -> every warp folds the 32 counts itself
    // (two barriers per bit, no serialised atomics; the two count buffers alternate so no third barrier is needed)
    uint32_t prefix = 0;
    for (int bit = 31; bit >= low_bit; --bit) {
        const uint32_t cand = prefix | (1u << bit);
        int cnt = 0;
        for (int i = beg; i < end; ++i) cnt += (keys[i] >= cand);
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        int* buf = sh + 40 + 32 * (bit & 1);
        if (lane == 0) buf[warp] = cnt;
        __syncthreads();
        const int total = __reduce_add_sync(0xffffffffu, buf[lane]);
        if (total >= keep) prefix = cand;
    }
    __syncthreads();
    // skipped low bits: the radix transform sets them to ones for negative values (and for NaN), to zeros otherwise
    if (low_bit > 0 && (!(prefix & 0x80000000u) || (prefix >> low_bit) == (0xffffffffu >> low_bit)))
        prefix |= (1u << low_bit) - 1u;
    // per-thread counts of greater / equal keys, block exclusive scans
    int gt = 0, eq = 0;
    for (int i = beg; i < end; ++i) { gt += (keys[i] > prefix); eq += (keys[i] == prefix); }
    auto block_excl_scan = [&](int v, int& total) {
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += n;
        }
        __syncthreads();
        if (lane == 31) sh[1 + warp] = inc;
        __syncthreads();
        if (warp == 0) {
            int w = sh[1 + lane], winc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int n = __shfl_up_sync(0xffffffffu, winc, o);
                if (lane >= o) winc += n;
            }
            sh[1 + lane] = winc - w;
            if (lane == 31) sh[33] = winc;
        }
        __syncthreads();
        total = sh[33];
        return sh[1 + warp] + inc - v;
    };
    int gt_total, eq_total;
    const int gt_before = block_excl_scan(gt, gt_total);
    const int eq_before = block_excl_scan(eq, eq_total);
    const int need = keep - gt_total;                          // equal keys to take, lowest index first
    const int eq_taken_before = min(eq_before, need);
    int slot = gt_before + eq_taken_before;
    int eq_seen = eq_before;
    for (int i = beg; i < end; ++i) {
        const uint32_t k = keys[i];
        bool take = k > prefix;
        if (k == prefix) { take = eq_seen < need; ++eq_seen; }
        if (take) out_idx[slot++] = i;
    }
}

__device__ __forceinline__ void pivot_select_body(const __nv_bfloat16* __restrict__ head_scores, int KVH, int L,
                                                  const uint8_t* __restrict__ keymask, int keep, int32_t* __restrict__ keep_idx,
                                                  __nv_bfloat16* __restrict__ score_out, const long long* __restrict__ tpos,
                                                  long long* __restrict__ tmin_out) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint32_t* keys = reinterpret_cast<uint32_t*>(smem);        // [L]
    int* sh = reinterpret_cast<int*>(smem + (size_t)L * 4);    // scratch
    const float rcp = 1.0f / (float)KVH;
    for (int i = threadIdx.x; i < L; i += blockDim.x) {
        // ATen mean(0): 4 accumulators over the reduced dim, folded ((v0+v1)+v2)+v3, times fp32(1/KVH)
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        for (int j = 0; j < KVH; ++j) v[j & 3] += __bfloat162float(head_scores[(size_t)j * L + i]);
        const __nv_bfloat16 s = __float2bfloat16_rn((((v[0] + v[1]) + v[2]) + v[3]) * rcp);
        if (score_out) score_out[i] = s;
        const float f = (keymask && keymask[i]) ? 1.0f : __bfloat162float(s);
        keys[i] = f32_to_ordered(f);
    }
    __syncthreads();
    block_select_top(keys, L, keep, keep_idx, sh, 16);        // bf16 scores: the low 16 key bits are zero
    if (tmin_out) {
        // smallest temporal position among the kept tokens (longvideo_cache.py:291) for the fused compaction
        __syncthreads();
        long long* smin = reinterpret_cast<long long*>((reinterpret_cast<uintptr_t>(sh) + 7) & ~(uintptr_t)7);
        long long mn = LLONG_MAX;
        for (int j = threadIdx.x; j < keep; j += blockDim.x) mn = min(mn, tpos[keep_idx[j]]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        if ((threadIdx.x & 31) == 0) smin[threadIdx.x >> 5] = mn;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); ++w) mn = min(mn, smin[w]);
            *tmin_out = mn;
        }
    }
}

// ---- peer exchange of the per-KV-head score rows (KV-head split of one video, SURVEY.md 8e): NVLink P2P stores from a
//      one-CTA kernel, a release store of the epoch into a flag word on every rank, an acquire spin in the select kernel
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// threads [0, n) each wait for one rank's flag to show `epoch`.  A peer that never arrives (crashed process, diverged
// control flow) must not hang the GPU for good: after `timeout_ns` (0 = wait for ever) the launch traps, which the host
// sees as a CUDA error at its next synchronisation.
__device__ __forceinline__ void xchg_wait(const uint32_t* flags, int n, uint32_t epoch, unsigned long long timeout_ns) {
    if ((int)threadIdx.x < n) {
        const unsigned long long t0 = globaltimer_ns();
        while (ld_acquire_sys(flags + threadIdx.x) != epoch) {
            __nanosleep(64);
            if (timeout_ns && globaltimer_ns() - t0 > timeout_ns) __trap();
        }
    }
    __syncthreads();
}
// one CTA per layer of the chunk stores this rank's rows into every peer's buffer (dst[layer][rank]: skipped), a one-CTA
// kernel behind it raises the flags
struct XchgPutBatch {
    const __nv_bfloat16* src[kMaxBatchLayers];
    __nv_bfloat16* dst[kMaxBatchLayers][8];
    long long n;                     // bf16 elements per layer
    int world, rank;
};
__global__ void __launch_bounds__(1024)
pivot_xchg_put_batch_kernel(const __grid_constant__ XchgPutBatch p) {
    pdl_enter();
    const int layer = blockIdx.x;
    const __nv_bfloat16* src = p.src[layer];
    for (int r = 0; r < p.world; ++r) {
        if (r == p.rank) continue;
        __nv_bfloat16* dst = p.dst[layer][r];
        if ((((uintptr_t)src | (uintptr_t)dst) & 15u) == 0) {
            const long long nv = p.n >> 3;
            for (long long i = threadIdx.x; i < nv; i += blockDim.x)
                reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(src)[i];
            for (long long i = (nv << 3) + threadIdx.x; i < p.n; i += blockDim.x) dst[i] = src[i];
        } else {
            for (long long i = threadIdx.x; i < p.n; i += blockDim.x) dst[i] = src[i];
        }
    }
    __threadfence_system();
}
struct XchgFlags {
    uint32_t* flags[8];
    int world, rank;
    uint32_t epoch;
};
__global__ void __launch_bounds__(32)
pivot_xchg_flag_kernel(XchgFlags p) {
    pdl_enter();                     // every CTA of the put kernel has completed (and fenced its peer stores)
    __threadfence_system();
    if ((int)threadIdx.x < p.world) st_release_sys(p.flags[threadIdx.x] + p.rank, p.epoch);
}

__global__ void __launch_bounds__(kSelThreads)
pivot_select_kernel(const __nv_bfloat16* __restrict__ head_scores, int KVH, int L, const uint8_t* __restrict__ keymask,
                    int keep, int32_t* __restrict__ keep_idx, __nv_bfloat16* __restrict__ score_out) {
    pdl_enter();
    pivot_select_body(head_scores, KVH, L, keymask, keep, keep_idx, score_out, nullptr, nullptr);
}

// one CTA per layer of the chunk
__global__ void __launch_bounds__(kSelThreads)
pivot_select_batch_kernel(const __grid_constant__ BatchLayers t, int KVH, int L, int keep, int reforge, long long* __restrict__ tmin,
                          const uint32_t* __restrict__ wait_flags, int wait_n, uint32_t wait_epoch, unsigned long long wait_ns) {
    pdl_enter();
    // rows of the other ranks arrive over NVLink: nothing of head_scores is read before every rank's flag is up
    if (wait_flags) xchg_wait(wait_flags, wait_n, wait_epoch, wait_ns);
    const int layer = blockIdx.x;
    pivot_select_body(t.head_scores[layer], KVH, L, t.keymask[layer], keep, t.keep_idx[layer], nullptr,
                      reforge ? t.pos[layer] : nullptr, reforge ? tmin + layer : nullptr);
}

// ======================================================================================= B3: compaction
// grid.x blocks gather KV rows (one 16-byte vector per thread-iteration); the LAST block handles positions.
struct CompactParams {
    int KVH, L, D, keep, n_pos, reforge;
    long long stride_h, stride_l, out_stride_h;
    long long v_stride_h, v_stride_l;
    long long pos_out_stride; // row stride of pos_out (= keep for a standalone [n_pos, keep] tensor)
    float ratio;              // fp32(keep / L)
};

__global__ void __launch_bounds__(256)
pivot_compact_kernel(const __nv_bfloat16* __restrict__ k, const __nv_bfloat16* __restrict__ v,
                     const int32_t* __restrict__ keep_idx, __nv_bfloat16* __restrict__ k_out,
                     __nv_bfloat16* __restrict__ v_out, const long long* __restrict__ pos,
                     long long* __restrict__ pos_out, CompactParams p) {
    pdl_enter();
    if (blockIdx.x == gridDim.x - 1) {
        if (!pos) return;
        __shared__ long long smin[32];
        const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
        for (int r = p.reforge ? 1 : 0; r < p.n_pos; ++r)
            for (int j = tid; j < p.keep; j += blockDim.x) pos_out[(size_t)r * p.keep + j] = pos[(size_t)r * p.L + keep_idx[j]];
        if (!p.reforge) return;
        long long mn = LLONG_MAX;
        for (int j = tid; j < p.keep; j += blockDim.x) mn = min(mn, pos[keep_idx[j]]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        if (lane == 0) smin[warp] = mn;
        __syncthreads();
        mn = smin[0];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) mn = min(mn, smin[w]);
        // m + ((p - m) * ratio).long(): int64 tensor times python float -> fp32 product, truncation toward zero
        for (int j = tid; j < p.keep; j += blockDim.x) {
            const float d = (float)(pos[keep_idx[j]] - mn);
            pos_out[j] = mn + (long long)(d * p.ratio);
        }
        return;
    }
    const int vec_per_row = p.D >> 3;
    const long long total = (long long)p.KVH * p.keep * vec_per_row;
    const long long nthreads = (long long)(gridDim.x - 1) * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += nthreads) {
        const int c = (int)(i % vec_per_row);
        const long long hj = i / vec_per_row;
        const int j = (int)(hj % p.keep);
        const int h = (int)(hj / p.keep);
        const int src_row = keep_idx[j];
        const size_t so = (size_t)h * p.stride_h + (size_t)src_row * p.stride_l + (size_t)c * 8;
        const size_t sv = (size_t)h * p.v_stride_h + (size_t)src_row * p.v_stride_l + (size_t)c * 8;
        const size_t dof = (size_t)h * p.out_stride_h + (size_t)j * p.D + (size_t)c * 8;
        if (k) *reinterpret_cast<uint4*>(k_out + dof) = __ldg(reinterpret_cast<const uint4*>(k + so));
        if (v) *reinterpret_cast<uint4*>(v_out + dof) = __ldg(reinterpret_cast<const uint4*>(v + sv));
    }
}

// Fused tail of an update (fast path): one CTA per kept token gathers its K and V rows of every KV head, writes its
// (re-indexed) position ids and - when re-forging - rotates K to the new position with the cos/sin row built in place.
// Replaces pivot_compact_kernel + pivot_rope_table_kernel + pivot_rope_kernel (longvideo_cache.py:278-306).
__device__ __forceinline__ void compact_rope_body(const __nv_bfloat16* __restrict__ k, const __nv_bfloat16* __restrict__ v,
                                                  const int32_t* __restrict__ keep_idx, __nv_bfloat16* __restrict__ k_out,
                                                  __nv_bfloat16* __restrict__ v_out, const long long* __restrict__ pos,
                                                  long long* __restrict__ pos_out, const long long* __restrict__ tmin,
                                                  const float* __restrict__ inv_freq, float scaling, const CompactParams& p,
                                                  const RopeParams& rp, int rotate) {
    __shared__ float s_cos[256], s_sin[256];
    __shared__ long long s_pos[3];
    const int j = blockIdx.x, tid = threadIdx.x;
    const int src_row = keep_idx[j];
    if (pos && tid < p.n_pos) {
        long long pv = pos[(size_t)tid * p.L + src_row];
        if (p.reforge && tid == 0) {
            // m + ((p - m) * ratio).long(): int64 tensor times python float -> fp32 product, truncation toward zero
            const long long mn = *tmin;
            pv = mn + (long long)((float)(pv - mn) * p.ratio);
        }
        pos_out[(size_t)tid * p.pos_out_stride + j] = pv;
        s_pos[tid] = pv;
    }
    const int vec_per_row = p.D >> 3;
    // V rows (and K rows when nothing is rotated): plain 16-byte copies
    for (int t = tid; t < p.KVH * vec_per_row; t += blockDim.x) {
        const int c = t % vec_per_row, h = t / vec_per_row;
        const size_t dof = (size_t)h * p.out_stride_h + (size_t)j * p.D + (size_t)c * 8;
        *reinterpret_cast<uint4*>(v_out + dof) =
            __ldg(reinterpret_cast<const uint4*>(v + (size_t)h * p.v_stride_h + (size_t)src_row * p.v_stride_l + (size_t)c * 8));
        if (!rotate)
            *reinterpret_cast<uint4*>(k_out + dof) =
                __ldg(reinterpret_cast<const uint4*>(k + (size_t)h * p.stride_h + (size_t)src_row * p.stride_l + (size_t)c * 8));
    }
    if (!rotate) return;
    __syncthreads();
    if (tid < p.D) rope_table_entry(rp, inv_freq, s_pos, tid, scaling, s_cos[tid], s_sin[tid]);
    __syncthreads();
    const int half = p.D >> 1, hv = half >> 3;
    for (int t = tid; t < p.KVH * hv; t += blockDim.x) {
        const int c0 = (t % hv) * 8, h = t / hv;
        const __nv_bfloat16* src = k + (size_t)h * p.stride_h + (size_t)src_row * p.stride_l;
        __nv_bfloat16* dst = k_out + (size_t)h * p.out_stride_h + (size_t)j * p.D;
        uint4 lo4 = *reinterpret_cast<const uint4*>(src + c0);
        uint4 hi4 = *reinterpret_cast<const uint4*>(src + c0 + half);
        const __nv_bfloat16* xl = reinterpret_cast<const __nv_bfloat16*>(&lo4);
        const __nv_bfloat16* xh = reinterpret_cast<const __nv_bfloat16*>(&hi4);
        uint4 ol4, oh4;
        __nv_bfloat16* ol = reinterpret_cast<__nv_bfloat16*>(&ol4);
        __nv_bfloat16* oh = reinterpret_cast<__nv_bfloat16*>(&oh4);
#pragma unroll
        for (int e = 0; e < 8; ++e)
            rope_rotate_pair(__bfloat162float(xl[e]), __bfloat162float(xh[e]), s_cos[c0 + e], s_sin[c0 + e], s_cos[c0 + half + e],
                             s_sin[c0 + half + e], 1, 1.0f, ol[e], oh[e]);
        *reinterpret_cast<uint4*>(dst + c0) = ol4;
        *reinterpret_cast<uint4*>(dst + c0 + half) = oh4;
    }
}

// grid (keep, layers): kept rows of every layer of the chunk straight into their caches
__global__ void __launch_bounds__(128)
pivot_compact_rope_batch_kernel(const __grid_constant__ BatchLayers t, const long long* __restrict__ tmin,
                                const float* __restrict__ inv_freq, float scaling, CompactParams p, RopeParams rp, int rotate) {
    pdl_enter();
    const int layer = blockIdx.y;
    p.stride_h = t.k_stride_h[layer]; p.stride_l = t.k_stride_l[layer];
    p.v_stride_h = t.v_stride_h[layer]; p.v_stride_l = t.v_stride_l[layer];
    p.out_stride_h = t.out_stride_h[layer];
    p.pos_out_stride = t.pos_out_stride[layer];
    compact_rope_body(t.k[layer], t.v[layer], t.keep_idx[layer], t.k_out[layer], t.v_out[layer], t.pos[layer], t.pos_out[layer],
                      tmin + layer, inv_freq, scaling, p, rp, rotate);
}

// up to four strided [heads, rows, D] block copies in ONE launch (cache append of K and V + the deferred overwrite of the
// previous layer's chunk head by its kept rows); replaces four torch copy_ launches per update
struct CopyJobs {
    int n;
    const __nv_bfloat16* src[4];
    __nv_bfloat16* dst[4];
    int heads[4], rows[4];
    long long src_stride_h[4], src_stride_l[4], dst_stride_h[4], dst_stride_l[4];
    long long vec_end[4];          // exclusive prefix of 16-byte vectors over the jobs
    int D;
};

__global__ void __launch_bounds__(256)
kv_block_copy_kernel(CopyJobs j) {
    pdl_enter();
    const int vpr = j.D >> 3;
    const long long total = j.vec_end[j.n - 1];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        int k = 0;
        while (i >= j.vec_end[k]) ++k;
        const long long li = i - (k ? j.vec_end[k - 1] : 0);
        const int c = (int)(li % vpr);
        const long long hr = li / vpr;
        const int r = (int)(hr % j.rows[k]);
        const int h = (int)(hr / j.rows[k]);
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(j.src[k] + h * j.src_stride_h[k] + r * j.src_stride_l[k] + c * 8));
        *reinterpret_cast<uint4*>(j.dst[k] + h * j.dst_stride_h[k] + r * j.dst_stride_l[k] + c * 8) = v;
    }
}

long long g_launches = 0;
// RTK_NO_KEY_ELISION=1 (or rtk_debug_key_elision(0)): score key patches like every other key - for A/B runs and debugging;
// the kept indices do not change
static int g_key_elision = -1;
bool key_elision_enabled() {
    if (g_key_elision < 0) {
        const char* e = getenv("RTK_NO_KEY_ELISION");
        g_key_elision = (e && e[0] == '1') ? 0 : 1;
    }
    return g_key_elision != 0;
}
// how long a select kernel waits for its peers' score rows before it traps (RTK_XCHG_TIMEOUT_S, default 120; 0 = for ever)
unsigned long long xchg_timeout_ns() {
    static const unsigned long long ns = [] {
        const char* e = getenv("RTK_XCHG_TIMEOUT_S");
        const double s = (e && e[0]) ? atof(e) : 120.0;
        return s > 0.0 ? (unsigned long long)(s * 1e9) : 0ull;
    }();
    return ns;
}
bool pdl_enabled() {
    static const bool on = [] {
        const char* e = getenv("RTK_NO_PDL");
        return !(e && e[0] && e[0] != '0');
    }();
    return on;
}

}  // namespace rtk

using namespace rtk;

extern "C" int rtk_version(void) { return RTK_ABI_VERSION; }

extern "C" int rtk_debug_key_elision(int on) {
    const int prev = rtk::key_elision_enabled() ? 1 : 0;
    if (on >= 0) rtk::g_key_elision = on ? 1 : 0;
    return prev;
}

#ifndef RTK_BUILD_ID
#define RTK_BUILD_ID "unknown"
#endif
extern "C" const char* rtk_build_id(void) { return RTK_BUILD_ID; }

extern "C" int64_t rtk_launch_count(void) { return (int64_t)rtk::g_launches; }

extern "C" const char* rtk_error_string(int code) {
    if (code == 0) return "ok";
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    switch (code) {
        case RTK_E_BADARG: return "rtk: bad argument (null pointer or non-positive size)";
        case RTK_E_ALIGN: return "rtk: pointer or stride not 16-byte aligned";
        case RTK_E_UNSUPPORTED: return "rtk: shape outside the supported envelope";
        case RTK_E_WORKSPACE: return "rtk: workspace too small";
        case RTK_E_DRIVER: return "rtk: cuTensorMapEncodeTiled unavailable or failed";
        default: return "rtk: unknown error";
    }
}

// pivot_rope_kernel over the p.heads rows of x and the p.heads2 rows of p.x2
static int rope_launch(const void* x, const void* cos, const void* sin, void* out, const RopeParams& p, cudaStream_t st) {
    const long long total = (long long)(p.heads + p.heads2) * p.L * (p.D / 16);
    long long grid = (total + 255) / 256;
    if (grid > 148 * 16) grid = 148 * 16;
    RTK_LAUNCH_PDL(pivot_rope_kernel, (unsigned)grid, 256, 0, st, (const __nv_bfloat16*)x, (const __nv_bfloat16*)cos, (const __nv_bfloat16*)sin, (__nv_bfloat16*)out, p);
    return 0;
}

extern "C" int rtk_pivot_rope(const void* x, int64_t heads, int64_t L, int64_t D, int64_t stride_h, int64_t stride_l,
                              const void* cos, const void* sin, int n_pos, const int32_t* mrope_section_host,
                              float inv_scale2, int forward, void* out, int64_t out_stride_h, int64_t out_stride_l,
                              void* stream) {
    RTK_NVTX("rtk_pivot_rope");
    if (!x || !cos || !sin || !out || heads < 1 || L < 1 || D < 16) return RTK_E_BADARG;
    if (D % 16 != 0 || (n_pos != 1 && n_pos != 3)) return RTK_E_UNSUPPORTED;
    if (n_pos == 3 && !mrope_section_host) return RTK_E_BADARG;
    if ((((uintptr_t)x | (uintptr_t)out) & 15u) != 0) return RTK_E_ALIGN;
    if ((stride_h | stride_l | out_stride_h | out_stride_l) % 8 != 0) return RTK_E_ALIGN;
    RopeParams p;
    p.heads = (int)heads; p.L = (int)L; p.D = (int)D; p.n_pos = n_pos; p.forward = forward;
    p.stride_h = stride_h; p.stride_l = stride_l; p.out_stride_h = out_stride_h; p.out_stride_l = out_stride_l;
    p.inv_scale2 = inv_scale2;
    p.heads2 = 0; p.x2 = nullptr; p.out2 = nullptr;
    p.stride_h2 = p.stride_l2 = p.out_stride_h2 = p.out_stride_l2 = 0;
    if (!mrope_bounds(n_pos, mrope_section_host, D, p.bound)) return RTK_E_UNSUPPORTED;
    return rope_launch(x, cos, sin, out, p, (cudaStream_t)stream);
}

extern "C" int rtk_pivot_select(const void* head_scores, int64_t KVH, int64_t L, const uint8_t* keymask, int64_t keep,
                                int32_t* keep_idx, void* score_out, void* stream) {
    RTK_NVTX("rtk_pivot_select");
    if (!head_scores || !keep_idx || KVH < 1 || L < 1 || keep < 1 || keep > L) return RTK_E_BADARG;
    if (L > 16384) return RTK_E_UNSUPPORTED;
    const size_t smem = (size_t)L * 4 + 112 * 4;
    cudaError_t e = cudaFuncSetAttribute(pivot_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    RTK_LAUNCH_PDL(pivot_select_kernel, 1, kSelThreads, smem, (cudaStream_t)stream, (const __nv_bfloat16*)head_scores, (int)KVH,
                   (int)L, keymask, (int)keep, keep_idx, (__nv_bfloat16*)score_out);
    return 0;
}

extern "C" int rtk_pivot_compact(const void* k, const void* v, int64_t KVH, int64_t L, int64_t D, int64_t stride_h,
                                 int64_t stride_l, const int32_t* keep_idx, int64_t keep, void* k_out, void* v_out,
                                 int64_t out_stride_h, const int64_t* pos, int n_pos, int64_t* pos_out, int reforge,
                                 void* stream) {
    RTK_NVTX("rtk_pivot_compact");
    if ((!k && !v) || !keep_idx || (k && !k_out) || (v && !v_out) || KVH < 1 || L < 1 || D < 8 || keep < 1 || keep > L)
        return RTK_E_BADARG;
    if (pos && (!pos_out || n_pos < 1)) return RTK_E_BADARG;
    if (D % 8 != 0) return RTK_E_UNSUPPORTED;
    if ((((uintptr_t)k | (uintptr_t)v | (uintptr_t)k_out | (uintptr_t)v_out) & 15u) != 0) return RTK_E_ALIGN;   // NULL passes
    if ((stride_h | stride_l | out_stride_h) % 8 != 0) return RTK_E_ALIGN;
    CompactParams p;
    p.KVH = (int)KVH; p.L = (int)L; p.D = (int)D; p.keep = (int)keep; p.n_pos = n_pos; p.reforge = reforge;
    p.stride_h = stride_h; p.stride_l = stride_l; p.out_stride_h = out_stride_h;
    p.v_stride_h = stride_h; p.v_stride_l = stride_l;
    p.pos_out_stride = keep;
    p.ratio = (float)((double)keep / (double)L);
    const long long total = KVH * keep * (D / 8);
    long long grid = (total + 255) / 256;
    if (grid > 148 * 8) grid = 148 * 8;
    RTK_LAUNCH_PDL(pivot_compact_kernel, (unsigned)(grid + 1), 256, 0, (cudaStream_t)stream,  (const __nv_bfloat16*)k, (const __nv_bfloat16*)v, keep_idx, (__nv_bfloat16*)k_out, (__nv_bfloat16*)v_out, (const long long*)pos, (long long*)pos_out, p);
    return 0;
}

extern "C" int rtk_pivot_rope_tables(const int64_t* pos, int n_pos, int64_t L, int64_t D, const float* inv_freq,
                                     const int32_t* mrope_section_host, float attention_scaling, void* cos_out,
                                     void* sin_out, void* stream) {
    RTK_NVTX("rtk_pivot_rope_tables");
    if (!pos || !inv_freq || !cos_out || !sin_out || L < 1 || D < 2) return RTK_E_BADARG;
    if (D % 2 != 0 || (n_pos != 1 && n_pos != 3)) return RTK_E_UNSUPPORTED;
    if (n_pos == 3 && !mrope_section_host) return RTK_E_BADARG;
    RopeParams p;
    p.heads = 1; p.L = (int)L; p.D = (int)D; p.n_pos = n_pos; p.forward = 0;
    p.stride_h = p.stride_l = p.out_stride_h = p.out_stride_l = 0;
    p.heads2 = 0; p.x2 = nullptr; p.out2 = nullptr;
    p.stride_h2 = p.stride_l2 = p.out_stride_h2 = p.out_stride_l2 = 0;
    p.inv_scale2 = 1.0f;
    if (!mrope_bounds(n_pos, mrope_section_host, D, p.bound)) return RTK_E_UNSUPPORTED;
    long long grid = (L * D + 255) / 256;
    if (grid > 148 * 8) grid = 148 * 8;
    RTK_LAUNCH_PDL(pivot_rope_table_kernel, (unsigned)grid, 256, 0, (cudaStream_t)stream,  (const long long*)pos, inv_freq, p, attention_scaling, (__nv_bfloat16*)cos_out, (__nv_bfloat16*)sin_out);
    return 0;
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

extern "C" size_t rtk_pivot_update_batch_workspace_bytes(int64_t H, int64_t KVH, int64_t L, int64_t D, int64_t n_layers) {
    if (H < 1 || KVH < 1 || L < 1 || D < 1 || n_layers < 1) return 0;
    const size_t n = (size_t)(n_layers < kMaxBatchLayers ? n_layers : kMaxBatchLayers);
    return align256(rtk_pivot_score_workspace_bytes(H * (int64_t)n, L)) +
           n * (align256((size_t)H * L * D * 2) + align256((size_t)KVH * L * D * 2)) + align256(n * sizeof(long long)) + 256 +
           n * key_elide_bytes(KVH, L, D) + 256;
}

extern "C" size_t rtk_pivot_update_workspace_bytes(int64_t H, int64_t KVH, int64_t L, int64_t D) {
    return rtk_pivot_update_batch_workspace_bytes(H, KVH, L, D, 1);
}

#ifndef RTK_UNROT_TOKEN_MAJOR
#define RTK_UNROT_TOKEN_MAJOR 1     // un-rotated copies laid out [L, heads, D] like the attention's own tensors
#endif

// The update chain of one group of <= kMaxBatchLayers layers whose arguments update_check accepted: un-rotate, score,
// exchange, select, compact + rotate.
static int pivot_update_group(const rtk_pivot_update_args* a, int n, char* ws, cudaStream_t st) {
    const rtk_pivot_update_args& a0 = a[0];
    const int64_t H = a0.H, KVH = a0.KVH, L = a0.L, D = a0.D;
    const bool reforge = a0.reforge != 0;
    // Layout of the un-rotated Q / K copies.  With 28 layers they are 1 GB and go through HBM: token-major rows make every
    // CTA of the un-rotation kernel write one contiguous block (all heads of its tokens) instead of one 256-byte row per
    // head 1 MB apart; the scoring kernels take any (head, token) strides through their tensor maps.
    const int64_t uq_sh = RTK_UNROT_TOKEN_MAJOR ? D : L * D, uq_sl = RTK_UNROT_TOKEN_MAJOR ? H * D : D;
    const int64_t uk_sh = RTK_UNROT_TOKEN_MAJOR ? D : L * D, uk_sl = RTK_UNROT_TOKEN_MAJOR ? KVH * D : D;
    void* score_ws = ws;                ws += align256(rtk_pivot_score_workspace_bytes(H * n, L));
    char* qu0 = ws;                     ws += (size_t)n * align256((size_t)H * L * D * 2);
    char* ku0 = ws;                     ws += (size_t)n * align256((size_t)KVH * L * D * 2);
    long long* tmin = (long long*)ws;   ws += align256((size_t)n * sizeof(long long)) + 256;
    char* kc0 = ws;                     ws += (size_t)n * align256((size_t)KVH * L * D * 2);      // key elision: compact K copies,
    char* slot0 = ws;                   ws += (size_t)n * align256((size_t)L * 4);                //   slots,
    int32_t* nkeys_ws = (int32_t*)ws;                                                              //   counts

    BatchLayers t = {};
    ScoreBatch sb = {};
    sb.n = n; sb.H = H; sb.KVH = KVH; sb.L = L; sb.D = D;
    for (int i = 0; i < kMaxBatchLayers; ++i) {
        const rtk_pivot_update_args& x = a[i < n ? i : 0];       // unused slots repeat layer 0 (never dereferenced)
        char* qu = qu0 + (size_t)(i < n ? i : 0) * align256((size_t)H * L * D * 2);
        char* ku = ku0 + (size_t)(i < n ? i : 0) * align256((size_t)KVH * L * D * 2);
        t.q[i] = (const __nv_bfloat16*)x.q;       t.q_stride_h[i] = x.q_stride_h;     t.q_stride_l[i] = x.q_stride_l;
        t.k_in[i] = (const __nv_bfloat16*)x.k;    t.kin_stride_h[i] = x.k_stride_h;   t.kin_stride_l[i] = x.k_stride_l;
        t.qu[i] = (__nv_bfloat16*)qu;             t.ku[i] = (__nv_bfloat16*)ku;
        t.k[i] = reforge ? (const __nv_bfloat16*)ku : (const __nv_bfloat16*)x.k;
        t.k_stride_h[i] = reforge ? uk_sh : x.k_stride_h;
        t.k_stride_l[i] = reforge ? uk_sl : x.k_stride_l;
        t.v[i] = (const __nv_bfloat16*)x.v;       t.v_stride_h[i] = x.v_stride_h;     t.v_stride_l[i] = x.v_stride_l;
        t.pos[i] = (const long long*)x.pos;       t.keymask[i] = x.keymask;
        t.k_out[i] = (__nv_bfloat16*)x.k_out;     t.v_out[i] = (__nv_bfloat16*)x.v_out;
        t.out_stride_h[i] = x.out_stride_h;
        t.pos_out[i] = (long long*)x.pos_out;     t.pos_out_stride[i] = x.pos_out_stride > 0 ? x.pos_out_stride : x.keep;
        t.keep_idx[i] = x.keep_idx;               t.head_scores[i] = (const __nv_bfloat16*)x.head_scores;
        if (i < n) {
            sb.q[i] = reforge ? (const void*)qu : x.q;
            sb.k[i] = reforge ? (const void*)ku : x.k;
            sb.q_stride_h[i] = reforge ? uq_sh : x.q_stride_h;   sb.q_stride_l[i] = reforge ? uq_sl : x.q_stride_l;
            sb.k_stride_h[i] = reforge ? uk_sh : x.k_stride_h;   sb.k_stride_l[i] = reforge ? uk_sl : x.k_stride_l;
            sb.head_scores[i] = x.head_scores;
        }
    }
    RopeParams rp = {};
    rp.heads = (int)H; rp.L = (int)L; rp.D = (int)D; rp.n_pos = a0.n_pos; rp.forward = 0;
    rp.out_stride_h = uq_sh; rp.out_stride_l = uq_sl;
    rp.heads2 = (int)KVH; rp.out_stride_h2 = uk_sh; rp.out_stride_l2 = uk_sl;
    rp.inv_scale2 = a0.inv_scale2;
    mrope_bounds(a0.n_pos, a0.mrope_section, D, rp.bound);
    const bool xchg = a0.xchg_world > 1;
    const int64_t score_rows = a0.score_rows > 0 ? a0.score_rows : KVH;
    // (skip_score: the un-rotated copies of the preceding skip_select call are still in the workspace)
    if (reforge && !a0.skip_score) {
        if (a0.inv_freq) {
            RTK_LAUNCH_PDL(pivot_unrope_qk_batch_kernel, dim3((unsigned)((L + kUnropeTok - 1) / kUnropeTok), (unsigned)n), 256, 0, st, t, a0.inv_freq,
                           a0.attention_scaling, rp);
        } else {
            // opaque rotary callable (one layer): un-rotate with the cos / sin tables it returned
            rp.stride_h = a0.q_stride_h; rp.stride_l = a0.q_stride_l;
            rp.x2 = t.k_in[0]; rp.out2 = t.ku[0]; rp.stride_h2 = a0.k_stride_h; rp.stride_l2 = a0.k_stride_l;
            const int rc = rope_launch(a0.q, a0.cos, a0.sin, t.qu[0], rp, st);
            if (rc) return rc;
        }
    }
    if (!a0.skip_score) {
        bool any_mask = false;
        for (int i = 0; i < n; ++i) any_mask = any_mask || a[i].keymask != nullptr;
        if (any_mask && key_elision_enabled()) {
            // key patches keep score 1.0 whatever their column sum is: pass 2 only visits the other keys of every layer
            KeyElide ke = {};
            ke.L = (int)L; ke.KVH = (int)KVH; ke.D = (int)D; ke.n_keys = nkeys_ws;
            for (int i = 0; i < kMaxBatchLayers; ++i) {
                const int j = i < n ? i : 0;
                ke.keymask[i] = a[j].keymask;
                ke.slot[i] = (int32_t*)(slot0 + (size_t)j * align256((size_t)L * 4));
                ke.k[i] = t.k[j]; ke.k_stride_h[i] = t.k_stride_h[j]; ke.k_stride_l[i] = t.k_stride_l[j];
                ke.kc[i] = (__nv_bfloat16*)(kc0 + (size_t)j * align256((size_t)KVH * L * D * 2));
            }
            int rc = key_elide_prepare(ke, n, sb, st);
            if (rc) return rc;
        }
        if (a0.ev_score_begin) cudaEventRecord((cudaEvent_t)a0.ev_score_begin, st);
        int rc = pivot_score_batch(sb, score_ws, rtk_pivot_score_workspace_bytes(H * n, L), st);
        if (rc) return rc;
        if (a0.ev_score_end) cudaEventRecord((cudaEvent_t)a0.ev_score_end, st);
    }
    if (a0.skip_select) {
        if (xchg) {
            // every layer's rows into every peer's buffer (one CTA per layer), then the flags of the batch
            XchgPutBatch xp = {};
            xp.n = (long long)KVH * L; xp.world = a0.xchg_world; xp.rank = a0.xchg_rank;
            for (int i = 0; i < n; ++i) {
                xp.src[i] = (const __nv_bfloat16*)a[i].head_scores;
                for (int r = 0; r < a0.xchg_world; ++r)
                    xp.dst[i][r] = (__nv_bfloat16*)a[i].xchg_scores[r] + (size_t)a0.xchg_rank * KVH * L;
            }
            RTK_LAUNCH_PDL(pivot_xchg_put_batch_kernel, (unsigned)n, 1024, 0, st, xp);
            XchgFlags xf = {};
            xf.world = a0.xchg_world; xf.rank = a0.xchg_rank; xf.epoch = a0.xchg_epoch;
            for (int r = 0; r < a0.xchg_world; ++r) xf.flags[r] = a0.xchg_flags[r];
            RTK_LAUNCH_PDL(pivot_xchg_flag_kernel, 1, 32, 0, st, xf);
        }
        return 0;
    }
    {
        const size_t smem = (size_t)L * 4 + 112 * 4;
        cudaError_t e = cudaFuncSetAttribute(pivot_select_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        RTK_LAUNCH_PDL(pivot_select_batch_kernel, (unsigned)n, kSelThreads, smem, st, t, (int)score_rows, (int)L, (int)a0.keep,
                       reforge ? 1 : 0, tmin, (const uint32_t*)(xchg ? a0.xchg_flags[a0.xchg_rank] : nullptr),
                       xchg ? a0.xchg_world : 0, a0.xchg_epoch, xchg_timeout_ns());
    }
    {
        // K (the un-rotated copy when re-forging), V, positions and - with inv_freq - the forward rotation at the
        // re-indexed positions; with cos / sin tables the caller rotates the kept keys itself (rtk_pivot_rope)
        CompactParams p = {};
        p.KVH = (int)KVH; p.L = (int)L; p.D = (int)D; p.keep = (int)a0.keep; p.n_pos = a0.pos ? a0.n_pos : 0; p.reforge = a0.reforge;
        p.ratio = (float)((double)a0.keep / (double)L);
        RopeParams rq = {};
        rq.D = (int)D; rq.n_pos = a0.n_pos; rq.L = (int)a0.keep;
        for (int i = 0; i < 6; ++i) rq.bound[i] = rp.bound[i];
        RTK_LAUNCH_PDL(pivot_compact_rope_batch_kernel, dim3((unsigned)a0.keep, (unsigned)n), 128, 0, st, t, (const long long*)tmin,
                       a0.inv_freq, a0.attention_scaling, p, rq, (reforge && a0.inv_freq) ? 1 : 0);
    }
    return 0;
}

// Every argument of an update of n layers (one chunk), checked before anything is launched.  A call that skips a step
// is not checked for what only that step reads: the scoring reads q and k, the selection and compaction read keep, V,
// the outputs and - when nothing is re-forged - k.
static int update_check(const rtk_pivot_update_args* layers, int64_t n, const void* workspace, size_t workspace_bytes) {
    if (!layers || n < 1 || !workspace) return RTK_E_BADARG;
    const rtk_pivot_update_args& a0 = layers[0];
    const bool scores = !a0.skip_score, selects = !a0.skip_select, xchg = a0.xchg_world > 1;
    if (!scores && !selects) return RTK_E_BADARG;
    if (a0.H < 1 || a0.KVH < 1 || a0.L < 1 || (selects && (a0.keep < 1 || a0.keep > a0.L))) return RTK_E_BADARG;
    if (a0.L > 16384 || a0.D % 16 != 0 || a0.D > 256) return RTK_E_UNSUPPORTED;
    if (scores && ((a0.D != 64 && a0.D != 128) || a0.H % a0.KVH != 0 || a0.H > 256)) return RTK_E_UNSUPPORTED;   // pivot_score_batch
    if (xchg) {
        // one flag set per call: the exchange covers one group of layers
        if (n > kMaxBatchLayers) return RTK_E_UNSUPPORTED;
        if (a0.xchg_world > 8 || a0.xchg_rank < 0 || a0.xchg_rank >= a0.xchg_world || (scores && selects)) return RTK_E_BADARG;
    }
    // the cos / sin tables of an opaque rotary callable are those of one layer; a batch re-forges with inv_freq
    if (a0.reforge && !a0.inv_freq && n > 1) return RTK_E_UNSUPPORTED;
    // the mrope blocks are read by the un-rotation and, with inv_freq, by the compaction's forward rotation
    int bound[6];
    if (a0.reforge && (scores || a0.inv_freq) && !mrope_bounds(a0.n_pos, a0.mrope_section, a0.D, bound)) return RTK_E_UNSUPPORTED;
    if (((uintptr_t)workspace & 255u) != 0) return RTK_E_ALIGN;
    if (workspace_bytes < rtk_pivot_update_batch_workspace_bytes(a0.H, a0.KVH, a0.L, a0.D, n)) return RTK_E_WORKSPACE;
    for (int64_t i = 0; i < n; ++i) {
        const rtk_pivot_update_args& x = layers[i];
        if (!x.q || !x.k || !x.v || !x.k_out || !x.v_out || !x.keep_idx || !x.head_scores) return RTK_E_BADARG;
        if (x.H != a0.H || x.KVH != a0.KVH || x.L != a0.L || x.D != a0.D || x.keep != a0.keep || x.reforge != a0.reforge ||
            x.n_pos != a0.n_pos || x.inv_freq != a0.inv_freq || x.attention_scaling != a0.attention_scaling ||
            x.inv_scale2 != a0.inv_scale2 || x.skip_select != a0.skip_select || x.skip_score != a0.skip_score ||
            x.score_rows != a0.score_rows || x.xchg_world != a0.xchg_world || x.xchg_rank != a0.xchg_rank ||
            x.xchg_epoch != a0.xchg_epoch || (x.pos == nullptr) != (a0.pos == nullptr))
            return RTK_E_UNSUPPORTED;                                 // one chunk: the layers share shape and rotary
        for (int j = 0; j < 3; ++j)
            if (x.mrope_section[j] != a0.mrope_section[j]) return RTK_E_UNSUPPORTED;
        if (x.reforge && (!x.pos || !x.pos_out || (!x.inv_freq && (!x.cos || !x.sin)))) return RTK_E_BADARG;
        if (xchg) {
            for (int r = 0; r < a0.xchg_world; ++r)
                if (!x.xchg_scores[r] || !a0.xchg_flags[r]) return RTK_E_BADARG;
            // where the rows live is part of the protocol
            const char* own = (const char*)x.xchg_scores[a0.xchg_rank];
            if (a0.skip_score && (const char*)x.head_scores != own) return RTK_E_BADARG;
            if (a0.skip_select && (const char*)x.head_scores != own + (size_t)a0.xchg_rank * a0.KVH * a0.L * 2) return RTK_E_BADARG;
        }
        if (x.pos && (selects || x.reforge) && (!x.pos_out || x.n_pos < 1 || x.n_pos > 3)) return RTK_E_BADARG;
        uintptr_t ptrs = 0;
        int64_t strides = 0;
        if (scores) {
            ptrs |= (uintptr_t)x.q;
            strides |= x.q_stride_h | x.q_stride_l;
        }
        if (scores || !x.reforge) {
            ptrs |= (uintptr_t)x.k;
            strides |= x.k_stride_h | x.k_stride_l;
        }
        if (selects) {
            ptrs |= (uintptr_t)x.v | (uintptr_t)x.k_out | (uintptr_t)x.v_out;
            strides |= x.v_stride_h | x.v_stride_l | x.out_stride_h;
        }
        if ((ptrs & 15u) != 0 || strides % 8 != 0) return RTK_E_ALIGN;
    }
    return 0;
}

extern "C" int rtk_pivot_update(const rtk_pivot_update_args* a, void* stream) {
    RTK_NVTX("rtk_pivot_update");
    if (!a) return RTK_E_BADARG;
    const int rc = update_check(a, 1, a->workspace, a->workspace_bytes);
    if (rc) return rc;
    return pivot_update_group(a, 1, (char*)a->workspace, (cudaStream_t)stream);
}

extern "C" int rtk_pivot_update_batch(const rtk_pivot_update_args* layers, int64_t n_layers, void* workspace,
                                      size_t workspace_bytes, void* stream) {
    RTK_NVTX("rtk_pivot_update_batch");
    int rc = update_check(layers, n_layers, workspace, workspace_bytes);
    if (rc) return rc;
    for (int64_t i = 0; i < n_layers; i += kMaxBatchLayers) {
        const int n = (int)((n_layers - i) < kMaxBatchLayers ? (n_layers - i) : kMaxBatchLayers);
        rc = pivot_update_group(layers + i, n, (char*)workspace, (cudaStream_t)stream);
        if (rc) return rc;
    }
    return 0;
}

extern "C" int rtk_kv_block_copy(int n_jobs, const void* const* src, void* const* dst, const int64_t* heads, const int64_t* rows,
                                 const int64_t* src_stride_h, const int64_t* src_stride_l, const int64_t* dst_stride_h,
                                 const int64_t* dst_stride_l, int64_t D, void* stream) {
    RTK_NVTX("rtk_kv_block_copy");
    if (n_jobs < 1 || n_jobs > 4 || !src || !dst || !heads || !rows || D < 8) return RTK_E_BADARG;
    if (D % 8 != 0) return RTK_E_UNSUPPORTED;
    CopyJobs j;
    j.n = n_jobs;
    j.D = (int)D;
    long long acc = 0;
    for (int k = 0; k < n_jobs; ++k) {
        if (!src[k] || !dst[k] || heads[k] < 1 || rows[k] < 0) return RTK_E_BADARG;
        if ((((uintptr_t)src[k] | (uintptr_t)dst[k]) & 15u) != 0) return RTK_E_ALIGN;
        if ((src_stride_h[k] | src_stride_l[k] | dst_stride_h[k] | dst_stride_l[k]) % 8 != 0) return RTK_E_ALIGN;
        j.src[k] = (const __nv_bfloat16*)src[k];
        j.dst[k] = (__nv_bfloat16*)dst[k];
        j.heads[k] = (int)heads[k];
        j.rows[k] = (int)rows[k];
        j.src_stride_h[k] = src_stride_h[k]; j.src_stride_l[k] = src_stride_l[k];
        j.dst_stride_h[k] = dst_stride_h[k]; j.dst_stride_l[k] = dst_stride_l[k];
        acc += heads[k] * rows[k] * (D / 8);
        j.vec_end[k] = acc;
    }
    for (int k = n_jobs; k < 4; ++k) j.vec_end[k] = acc;
    if (acc == 0) return 0;
    long long grid = (acc + 255) / 256;
    if (grid > 148 * 8) grid = 148 * 8;
    RTK_LAUNCH_PDL(kv_block_copy_kernel, (unsigned)grid, 256, 0, (cudaStream_t)stream, j);
    return 0;
}
