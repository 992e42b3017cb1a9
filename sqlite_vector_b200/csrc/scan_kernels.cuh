// scan_kernels.cuh — sm_100a kernels of the single-query (HBM-bound) distance scan.
//
// Replaces, for a whole resident shard at once, the per-row loop of the reference:
//   fn = dispatch_distance_table[metric][type]; d = fn(q,row,dim); clamp; slot update
//   (/root/reference/src/sqlite-vector.c:2089-2107 and :2138-2153, kernels in src/distance-cpu.c:39-693).
//
// Design (see DESIGN.md §3):
//   * corpus rows are dense in HBM ([n][pitch], pitch = dim*elt rounded up to 16 B, zero padded);
//   * every WARP owns a contiguous range of rows ("stream") and pulls it through its own ring of
//     shared-memory stages with TMA bulk copies (cp.async.bulk + mbarrier complete_tx) that it issues
//     itself — no block-level barrier anywhere in the steady state;
//   * P = 1..32 lanes cooperate on a row; 16-byte LDS with a per-row rotation keeps the shared-memory
//     reads conflict-free; integer types use dp4a / vabsdiff4 (exact int32), fp types FFMA;
//   * top-k: each warp keeps the k smallest distances of its own stream in shared memory and logs every
//     row that beats the running k-th value (strict <).  That log is a superset of the rows that can
//     ever enter the reference's k slots; filter_kernel tightens it with prefix thresholds and the
//     host replays the reference's slot algorithm over the few hundred survivors, which reproduces
//     the reference's history-dependent tie handling exactly.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

namespace vsb {

constexpr int kWarps = 8;             // consumer warps per CTA (each one is a stream)
constexpr int kThreads = kWarps * 32;
constexpr int kMaxStages = 8;         // ring stages per warp
constexpr int kBarrierBytes = 1024;   // reserved at the start of dynamic smem for mbarriers + scalars

enum { T_F32 = 1, T_F16 = 2, T_BF16 = 3, T_U8 = 4, T_I8 = 5 };
enum { MC_L2 = 0, MC_COS = 1, MC_DOT = 2, MC_L1 = 3 };  // L2 and SQUARED_L2 share a kernel (root flag)

constexpr int kMaxGroup = 8;          // independent queries one launch can scan back to back

struct ScanQuery {        // per-query pointers of a launch
    const uint8_t *query; // device, pitch bytes, zero padded
    float *lists;         // k <= 32: [CTAs][32] the k smallest distances of each CTA's rows, sorted ascending, +INF padded;
                          // k > 32:  [streams][kcap] k smallest distances of each stream (unsorted)
    float *tlocal;        // k <= 32: [streams] k-th smallest distance over the EARLIER streams of the same CTA (+INF if < k rows)
    uint2 *logs;          // [streams][logcap] (dist bits, local row)
    int *counts;          // [streams] log entries written (may exceed logcap => overflow)
    int *ctrl;            // ctrl[1] = overflow flag
    float *dist_all;      // optional [n]
};

struct ScanParams {
    const uint8_t *vec;   // [n][pitch]
    long long n;
    int pitch;            // bytes per row (multiple of 16)
    int nc;               // 16-byte chunks per row
    int log2P;            // lanes per row = 1 << log2P
    int wtile_bytes;      // (32 >> log2P) * pitch
    int nsw;              // ring stages per warp
    int root;             // metric L2: take the square root
    int k;                // 0 => no top-k (dist_all only)
    int kcap;             // k rounded up to 32
    int logcap;
    int nq;               // queries scanned by this launch (1..kMaxGroup)
    ScanQuery q[kMaxGroup];
    // adaptive row partition (optional): bounds[c] .. bounds[c+1] are the warp-tiles of CTA c (contiguous, ascending, any
    // sizes: the exactness argument only needs streams to be contiguous row ranges in scan order).  Each CTA reports the
    // cycles it took; filter_kernel turns speeds into the partition of the query after next (SMs do not all pull from
    // HBM at the same rate, and with equal shares the slowest one sets the kernel time).
    const long long *bounds;   // [gridDim.x + 1] or nullptr (equal shares)
    unsigned *cta_time;        // [gridDim.x] or nullptr
};

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// TMA bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ uint4 ldg_stream(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// monotone float -> uint32 key (total order, -0 < +0), used for warp-wide max via REDUX
__device__ __forceinline__ uint32_t fkey(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// ------------------------------------------------------------------ accumulation
struct Accum {
    float s0, s1;   // fp: primary sum split in two chains (dot / sum of squares / sum of |d|)
    float ny;       // fp cosine: row norm (the query norm is computed once per query, QueryNorm)
    int ia, ib;     // int: dot or sad, row norm
};

template <int VT>
__device__ __forceinline__ void unpack8(const uint4 v, float (&o)[8]) {
    if constexpr (VT == T_F32) {
        o[0] = __uint_as_float(v.x); o[1] = __uint_as_float(v.y); o[2] = __uint_as_float(v.z); o[3] = __uint_as_float(v.w);
    } else if constexpr (VT == T_F16) {
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            __half2 h = *reinterpret_cast<const __half2 *>(&w[j]);
            float2 f = __half22float2(h);
            o[2 * j] = f.x; o[2 * j + 1] = f.y;
        }
    } else {  // bf16: value = bits << 16 (src/distance-cpu.h:100-102)
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            o[2 * j] = __uint_as_float(w[j] << 16);
            o[2 * j + 1] = __uint_as_float(w[j] & 0xFFFF0000u);
        }
    }
}

// one 16-byte chunk of the row (r) against the same chunk of the query (q)
template <int VT, int MC>
__device__ __forceinline__ void accum16(Accum &A, const uint4 r, const uint4 q) {
    if constexpr (VT == T_U8 || VT == T_I8) {
        const uint32_t rw[4] = {r.x, r.y, r.z, r.w}, qw[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if constexpr (MC == MC_L1) {
                // sum |a-b|: per-byte absolute difference, then dot with 1s (exact)
                uint32_t ad = (VT == T_U8) ? __vabsdiffu4(rw[j], qw[j]) : __vabsdiffs4(rw[j], qw[j]);
                A.ia = (int)__dp4a(ad, 0x01010101u, (uint32_t)A.ia);
            } else {
                if constexpr (VT == T_U8) {
                    A.ia = (int)__dp4a(rw[j], qw[j], (uint32_t)A.ia);
                    if constexpr (MC != MC_DOT) A.ib = (int)__dp4a(rw[j], rw[j], (uint32_t)A.ib);
                } else {
                    A.ia = __dp4a((int)rw[j], (int)qw[j], A.ia);
                    if constexpr (MC != MC_DOT) A.ib = __dp4a((int)rw[j], (int)rw[j], A.ib);
                }
            }
        }
    } else {
        constexpr int NE = (VT == T_F32) ? 4 : 8;
        float y[8], x[8];
        unpack8<VT>(r, y);
        unpack8<VT>(q, x);
        // Plain IEEE accumulation, no per-element special-value tests: the reference's NaN-lane / infinity policies (f16: all
        // metrics, src/distance-cpu.c:318-466; bf16 L2: :164-197) only matter for rows (or queries) that actually hold a NaN or
        // an infinity, and any such element leaves a non-finite accumulator behind.  Those rows are recomputed with the
        // reference's exact policy by special_row_distance (row_needs_exact below).
#pragma unroll
        for (int j = 0; j < NE; ++j) {
            float &s = (j & 1) ? A.s1 : A.s0;
            if constexpr (MC == MC_L2) {
                const float d = x[j] - y[j];
                s = fmaf(d, d, s);
            } else if constexpr (MC == MC_L1) {
                s += fabsf(x[j] - y[j]);
            } else if constexpr (MC == MC_DOT) {
                s = fmaf(x[j], y[j], s);
            } else {  // cosine
                s = fmaf(x[j], y[j], s);
                A.ny = fmaf(y[j], y[j], A.ny);
            }
        }
    }
}

struct QueryNorm {
    float f;     // fp: sum x^2 of the query
    int i;       // int: sum q^2 (bit pattern; unsigned for u8)
};

// accumulators -> the float the reference kernel returns, then the nearly-zero clamp
template <int VT, int MC>
__device__ __forceinline__ float finalize(const Accum &A, const QueryNorm qn, int root) {
    float d;
    if constexpr (VT == T_U8 || VT == T_I8) {
        if constexpr (MC == MC_L2) {
            // sum (a-b)^2 = |q|^2 + |row|^2 - 2 q.row, exact in 32-bit (src/distance-avx2.c int32 path;
            // equals the float-accumulating scalar kernel, src/distance-cpu.c:470-502, while sums < 2^24)
            float f;
            if constexpr (VT == T_U8) f = (float)((uint32_t)qn.i + (uint32_t)A.ib - 2u * (uint32_t)A.ia);
            else f = (float)(qn.i + A.ib - 2 * A.ia);
            d = root ? __fsqrt_rn(f) : f;
        } else if constexpr (MC == MC_COS) {
            // src/distance-cpu.c:533-538, 645-650
            if (qn.i == 0 || A.ib == 0) d = 1.0f;
            else {
                float fq = (VT == T_U8) ? (float)(uint32_t)qn.i : (float)qn.i;
                float fr = (VT == T_U8) ? (float)(uint32_t)A.ib : (float)A.ib;
                float fd = (VT == T_U8) ? (float)(uint32_t)A.ia : (float)A.ia;
                float den = __fmul_rn(__fsqrt_rn(fq), __fsqrt_rn(fr));
                d = __fsub_rn(1.0f, __fdiv_rn(fd, den));
            }
        } else if constexpr (MC == MC_DOT) {
            d = (VT == T_U8) ? -(float)(uint32_t)A.ia : -(float)A.ia;
        } else {
            d = (float)(uint32_t)A.ia;
        }
    } else {
        const float s = A.s0 + A.s1;
        if constexpr (MC == MC_L2) d = root ? __fsqrt_rn(s) : s;
        else if constexpr (MC == MC_DOT) d = -s;
        else if constexpr (MC == MC_L1) d = s;
        else {
            if constexpr (VT == T_F16) {
                // src/distance-cpu.c:457-465 (finite inputs; rows with NaN / Inf go through special_row_distance): bad
                // denominator -> 1; clamp cos to [-1,1]
                float den = __fmul_rn(__fsqrt_rn(qn.f), __fsqrt_rn(A.ny));
                if (!(den > 0.0f) || isinf(den) || den != den || isinf(s) || s != s) d = 1.0f;
                else {
                    float c = __fdiv_rn(s, den);
                    c = fminf(1.0f, fmaxf(-1.0f, c));
                    d = 1.0f - c;
                }
            } else {
                // src/distance-cpu.c:105-109, 248-252
                if (qn.f == 0.0f || A.ny == 0.0f) d = 1.0f;
                else d = __fsub_rn(1.0f, __fdiv_rn(s, __fmul_rn(__fsqrt_rn(qn.f), __fsqrt_rn(A.ny))));
            }
        }
    }
    // nearly_zero_float32: |d| <= 8*FLT_EPSILON -> +0.0 (src/sqlite-vector.c:994-996, 2099, 2143)
    return (fabsf(d) <= 8.0f * FLT_EPSILON) ? 0.0f : d;
}

// ------------------------------------------------------------------ rows with NaN / Inf elements (rare path)
// kinds whose reference kernel treats special values differently from IEEE propagation
template <int VT, int MC>
__host__ __device__ constexpr bool has_special_policy() { return VT == T_F16 || (VT == T_BF16 && MC == MC_L2); }

// after accum_reduce: does this row (or the query) hold a NaN / Inf?  (finite inputs cannot overflow these sums: f16 values
// are <= 65504 and bf16 L2 sums of finite differences stay finite up to ~1e19 per element)
template <int VT, int MC>
__device__ __forceinline__ bool row_needs_exact(const Accum &A, const QueryNorm qn) {
    if constexpr (!has_special_policy<VT, MC>()) return false;
    else if constexpr (MC == MC_COS) return !(fabsf(A.s0 + A.s1) <= FLT_MAX) || !(A.ny <= FLT_MAX) || !(qn.f <= FLT_MAX);
    else return !(fabsf(A.s0 + A.s1) <= FLT_MAX);
}

// The reference's own element loop for one row, one thread, element order (fp32 accumulation instead of double: the result
// classes — NaN, +Inf, -Inf, 1.0 — are exact, finite values agree to ~dim * 2^-24):
//   f16 L2 / L1 (:318-400): a lane with an infinity that is not paired with an equal-signed infinity -> +INF at once (checked
//       BEFORE the NaN test); NaN lanes skipped; Inf - Inf poisons the sum (LASSQ: NaN unless every other difference is 0)
//   f16 DOT (:402-432): NaN lanes skipped; the FIRST infinite product decides: -INF if positive, +INF if negative; Inf * 0 poisons
//   f16 COSINE (:434-466): NaN lanes skipped; any infinity -> 1; bad denominator / non-finite dot -> 1; clamp to [-1, 1]
//   bf16 L2 (:164-197): float difference; infinite difference -> +INF; NaN difference skipped
template <int VT, int MC>
__device__ __noinline__ float special_row_distance(const uint8_t *row, const uint8_t *query, int nelem, int root) {
    const uint16_t *yb = reinterpret_cast<const uint16_t *>(row), *xb = reinterpret_cast<const uint16_t *>(query);
    float s = 0.0f, nx = 0.0f, ny = 0.0f;
    bool poisoned = false, anynz = false;
    for (int e = 0; e < nelem; ++e) {
        float xf, yf;
        if constexpr (VT == T_F16) {
            xf = __half2float(__ushort_as_half(xb[e]));
            yf = __half2float(__ushort_as_half(yb[e]));
        } else {
            xf = __uint_as_float((uint32_t)xb[e] << 16);
            yf = __uint_as_float((uint32_t)yb[e] << 16);
        }
        if constexpr (VT == T_BF16) {                                           // bf16 L2
            const float d = xf - yf;
            if (isinf(d)) return INFINITY;
            if (d == d) s = fmaf(d, d, s);
        } else if constexpr (MC == MC_L2 || MC == MC_L1) {
            const bool xi = isinf(xf), yi = isinf(yf);
            if ((xi || yi) && !(xi && yi && (xf > 0.0f) == (yf > 0.0f))) return INFINITY;
            if (xf != xf || yf != yf) continue;
            const float d = xf - yf;                                            // NaN for an equal-signed pair of infinities
            if (d != d) poisoned = true;
            else {
                if (d != 0.0f) anynz = true;
                s = (MC == MC_L2) ? fmaf(d, d, s) : s + fabsf(d);
            }
        } else {
            if (xf != xf || yf != yf) continue;
            if constexpr (MC == MC_DOT) {
                const float p = xf * yf;                                        // exact for f16 inputs; infinite iff an input is
                if (isinf(p)) return p > 0.0f ? -INFINITY : INFINITY;
                s += p;                                                         // Inf * 0 = NaN poisons, like `dot += p`
            } else {
                if (isinf(xf) || isinf(yf)) return 1.0f;
                s = fmaf(xf, yf, s); nx = fmaf(xf, xf, nx); ny = fmaf(yf, yf, ny);
            }
        }
    }
    float d;
    if constexpr (MC == MC_L2) {
        if (poisoned) d = anynz ? __int_as_float(0x7FC00000) : 0.0f;           // LASSQ: scale == 0 -> 0 (:346 / :194)
        else d = root ? __fsqrt_rn(s) : s;
    } else if constexpr (MC == MC_L1) {
        d = poisoned ? __int_as_float(0x7FC00000) : s;
    } else if constexpr (MC == MC_DOT) {
        d = -s;
    } else {
        const float den = __fmul_rn(__fsqrt_rn(nx), __fsqrt_rn(ny));
        if (!(den > 0.0f) || isinf(den) || den != den || isinf(s) || s != s) d = 1.0f;
        else d = 1.0f - fminf(1.0f, fmaxf(-1.0f, __fdiv_rn(s, den)));
    }
    return (fabsf(d) <= 8.0f * FLT_EPSILON) ? 0.0f : d;
}

__device__ __forceinline__ void accum_reduce(Accum &A, int P) {
    for (int off = P >> 1; off >= 1; off >>= 1) {
        A.s0 += __shfl_xor_sync(0xFFFFFFFFu, A.s0, off);
        A.s1 += __shfl_xor_sync(0xFFFFFFFFu, A.s1, off);
        A.ny += __shfl_xor_sync(0xFFFFFFFFu, A.ny, off);
        A.ia += __shfl_xor_sync(0xFFFFFFFFu, A.ia, off);
        A.ib += __shfl_xor_sync(0xFFFFFFFFu, A.ib, off);
    }
}

// ------------------------------------------------------------------ warp-private k-smallest list
// list[0..kcap) in shared memory: entries < k start at +INF, entries >= k at -INF (never the max).
// Returns the current maximum (= running k-th smallest, +INF until k rows were seen) and its position.
__device__ __forceinline__ void list_argmax(const float *list, int kcap, int lane, float &thr, int &pos) {
    float best = list[lane];
    int bi = lane;
    for (int j = lane + 32; j < kcap; j += 32) {
        float v = list[j];
        if (v > best) { best = v; bi = j; }
    }
    uint32_t key = fkey(best);
    uint32_t mx = __reduce_max_sync(0xFFFFFFFFu, key);
    int src = __ffs(__ballot_sync(0xFFFFFFFFu, key == mx)) - 1;
    thr = __shfl_sync(0xFFFFFFFFu, best, src);
    pos = __shfl_sync(0xFFFFFFFFu, bi, src);
}

// bitonic sort of one value per lane, ascending by lane
__device__ __forceinline__ float warp_sort_asc(float v, int lane) {
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride >= 1; stride >>= 1) {
            const float o = __shfl_xor_sync(0xFFFFFFFFu, v, stride);
            const bool up = ((lane & size) == 0);            // ascending block?
            const bool lower = ((lane & stride) == 0);
            v = (lower == up) ? fminf(v, o) : fmaxf(v, o);
        }
    }
    return v;
}
// v is a bitonic sequence across the lanes -> ascending
__device__ __forceinline__ float warp_bitonic_merge_asc(float v, int lane) {
#pragma unroll
    for (int stride = 16; stride >= 1; stride >>= 1) {
        const float o = __shfl_xor_sync(0xFFFFFFFFu, v, stride);
        v = ((lane & stride) == 0) ? fminf(v, o) : fmaxf(v, o);
    }
    return v;
}

__device__ __forceinline__ float funkey(uint32_t k) {  // inverse of fkey
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

// k <= 32: the warp's k-list lives in one register per lane, SORTED ascending (lanes >= k hold +INF); the running
// k-th value is lane k-1.  Incoming lists are sorted too (scan_kernel publishes them that way), so an offer is either
// a couple of shift-inserts or one bitonic merge — no serial chain of k inserts for the first streams of a segment.
struct SortedList {
    float v, thr;
    int k;
    __device__ __forceinline__ void init(int lane, int k_) { k = k_; v = INFINITY; thr = INFINITY; }
    __device__ __forceinline__ void insert(int lane, float dv) {           // dv < thr
        const int pos = __popc(__ballot_sync(0xFFFFFFFFu, v <= dv));       // elements that stay in front of dv
        const float up = __shfl_up_sync(0xFFFFFFFFu, v, 1);
        v = (lane < pos) ? v : (lane == pos ? dv : up);
        if (lane >= k) v = INFINITY;
        thr = __shfl_sync(0xFFFFFFFFu, v, k - 1);
    }
    // val: a sorted ascending list, one value per lane, +INF padded
    __device__ __forceinline__ void offer_sorted(int lane, float val) {
        const int cnt = __popc(__ballot_sync(0xFFFFFFFFu, val < thr));     // these are the first cnt lanes
        if (cnt == 0) return;
        if (cnt <= 2) {
            const float a = __shfl_sync(0xFFFFFFFFu, val, 0);
            insert(lane, a);
            if (cnt == 2) {
                const float b = __shfl_sync(0xFFFFFFFFu, val, 1);
                if (b < thr) insert(lane, b);
            }
            return;
        }
        // 32 smallest of the 64 values: min(L[i], R[31-i]) is bitonic; one merge network sorts it
        const float rev = __shfl_sync(0xFFFFFFFFu, val, 31 - lane);
        v = warp_bitonic_merge_asc(fminf(v, rev), lane);
        if (lane >= k) v = INFINITY;
        thr = __shfl_sync(0xFFFFFFFFu, v, k - 1);
    }
};

// ------------------------------------------------------------------ the scan kernel
// One launch scans the shard for prm.nq independent queries back to back (nq = 1: the plain single-query call; nq > 1: a
// group submitted together by the sharded launcher).  Every CTA keeps its row range and simply starts the next query when
// its 8 streams are done: no kernel boundary, no launch gap, and the TMA ring runs across the query boundary (the first
// tiles of query g+1 are already in flight while the last tiles of query g are consumed).  Each query still has its own
// k-lists, logs, counters and control words: results are exactly those of nq separate launches.
template <int VT, int MC, bool DIRECT>
__global__ void __launch_bounds__(kThreads, 1) scan_kernel(const ScanParams prm) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem);                    // [kWarps][kMaxStages]
    uint8_t *qs = smem + kBarrierBytes;                                      // [2][pitch] query of the current / next scan
    const int list_bytes = kWarps * prm.kcap * 4;
    float *lists_s = reinterpret_cast<float *>(qs + 2 * prm.pitch);          // [2][kWarps][kcap]
    uint8_t *ring = qs + ((2 * prm.pitch + 2 * list_bytes + 127) & ~127);    // [kWarps][nsw][wtile_bytes]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int P = 1 << prm.log2P, rpw = 32 >> prm.log2P;
    const int nsw = prm.nsw;
    const long long clk0 = clock64();

    // ---- prologue: barriers, first query
    if (tid == 0) {
        for (int i = 0; i < kWarps * kMaxStages; ++i) mbar_init(&bars[i], 1);
        fence_barrier_init();
    }
    for (int i = tid; i < prm.nc; i += kThreads)
        reinterpret_cast<uint4 *>(qs)[i] = reinterpret_cast<const uint4 *>(prm.q[0].query)[i];
    __syncthreads();

    // ---- this warp's stream: a contiguous range of warp-tiles (rpw rows each), the same for every query of the launch
    const long long sidx = (long long)blockIdx.x * kWarps + warp;
    const long long T = (prm.n + rpw - 1) / rpw;
    long long c0, c1;                                                        // this CTA's warp-tiles
    if (prm.bounds != nullptr) { c0 = prm.bounds[blockIdx.x]; c1 = prm.bounds[blockIdx.x + 1]; }
    else { c0 = (T * blockIdx.x) / gridDim.x; c1 = (T * (blockIdx.x + 1)) / gridDim.x; }
    const long long t0 = c0 + ((c1 - c0) * warp) / kWarps, t1 = c0 + ((c1 - c0) * (warp + 1)) / kWarps;
    const int ntiles = (int)(t1 - t0);

    uint64_t *mybars = bars + warp * kMaxStages;
    uint8_t *myring = ring + (size_t)warp * nsw * prm.wtile_bytes;
    const uint64_t pol = policy_evict_first();

    // The warp consumes nq * ntiles tiles in all (its stream once per query); the ring simply keeps running across query
    // boundaries: the tile fetched into the stage just freed is always the one nsw positions ahead, which near the end of
    // a query is one of the first tiles of the next query.
    const unsigned total = (unsigned)prm.nq * (unsigned)ntiles;             // tiles this warp consumes in this launch
    unsigned fetched = 0;                                                    // tiles issued so far (lane 0)
    int pf_it = 0;                                                           // stream tile index of the next fetch
    auto issue = [&](int s) {  // lane 0 only: next tile of the sequence into stage s
        const long long row0 = (t0 + pf_it) * rpw;
        long long rows = prm.n - row0;
        if (rows > rpw) rows = rpw;
        const uint32_t bytes = (uint32_t)rows * (uint32_t)prm.pitch;
        mbar_expect_tx(&mybars[s], bytes);
        bulk_g2s(myring + (size_t)s * prm.wtile_bytes, prm.vec + (size_t)row0 * prm.pitch, bytes, &mybars[s], pol);
        ++fetched;
        if (++pf_it == ntiles) pf_it = 0;
    };
    if constexpr (!DIRECT) {
        if (lane == 0)
            for (int s = 0; s < nsw && fetched < total; ++s) issue(s);
    }
    int stage = 0;                                                           // ring position of the next tile to consume
    uint32_t parity = 0;

    const int r = lane >> prm.log2P, p = lane & (P - 1);
    const int cnt = (prm.nc > p) ? (prm.nc - p + P - 1) >> prm.log2P : 0;  // chunks owned by this lane
    const int i0 = cnt ? (r % cnt) : 0;                                       // rotation: conflict-free LDS.128
    const bool topk = prm.k > 0;
    constexpr bool kFix16 = has_special_policy<VT, MC>();   // rows with NaN / Inf are recomputed from the staged tile: see special_row_distance
    const uint8_t *fix_row = nullptr;
    int fix_stage = 0;

    for (int g = 0; g < prm.nq; ++g) {
        const ScanQuery &Q = prm.q[g];
        const uint8_t *qbuf = qs + (size_t)(g & 1) * prm.pitch;
        float *mylist = lists_s + ((size_t)(g & 1) * kWarps + warp) * prm.kcap;

        // query norm (every warp computes it the same way: lane-strided chunks, butterfly sum)
        QueryNorm qn;
        {
            float f = 0.0f;
            int iq = 0;
            for (int c = lane; c < prm.nc; c += 32) {
                const uint4 q = reinterpret_cast<const uint4 *>(qbuf)[c];
                if constexpr (VT == T_U8) {
                    iq = (int)__dp4a(q.x, q.x, (uint32_t)iq); iq = (int)__dp4a(q.y, q.y, (uint32_t)iq);
                    iq = (int)__dp4a(q.z, q.z, (uint32_t)iq); iq = (int)__dp4a(q.w, q.w, (uint32_t)iq);
                } else if constexpr (VT == T_I8) {
                    iq = __dp4a((int)q.x, (int)q.x, iq); iq = __dp4a((int)q.y, (int)q.y, iq);
                    iq = __dp4a((int)q.z, (int)q.z, iq); iq = __dp4a((int)q.w, (int)q.w, iq);
                } else {
                    float x[8];
                    unpack8<VT>(q, x);
                    constexpr int NE = (VT == T_F32) ? 4 : 8;
#pragma unroll
                    for (int j = 0; j < NE; ++j) f = fmaf(x[j], x[j], f);
                }
            }
            for (int off = 16; off >= 1; off >>= 1) {
                f += __shfl_xor_sync(0xFFFFFFFFu, f, off);
                iq += __shfl_xor_sync(0xFFFFFFFFu, iq, off);
            }
            qn.f = f; qn.i = iq;
        }
        for (int j = lane; j < prm.kcap; j += 32) mylist[j] = (j < prm.k) ? INFINITY : -INFINITY;
        __syncwarp();

        float thr = INFINITY;
        int pos = 0, logged = 0;
        uint2 *mylog = Q.logs + (size_t)sidx * prm.logcap;

        for (int it = 0; it < ntiles; ++it) {
            const long long row0 = (t0 + it) * rpw;
            const bool valid = (row0 + r) < prm.n;
            Accum A = {0.f, 0.f, 0.f, 0, 0};
            if constexpr (!DIRECT) {
                const int s = stage;
                mbar_wait(&mybars[s], parity);
                if (++stage == nsw) { stage = 0; parity ^= 1u; }
                const uint8_t *rowp = myring + (size_t)s * prm.wtile_bytes + (size_t)r * prm.pitch;
                if (valid) {
#pragma unroll 4
                    for (int i = 0; i < cnt; ++i) {
                        int ii = i0 + i;
                        if (ii >= cnt) ii -= cnt;
                        const int c = p + (ii << prm.log2P);
                        const uint4 rv = *reinterpret_cast<const uint4 *>(rowp + (size_t)c * 16);
                        const uint4 qv = *reinterpret_cast<const uint4 *>(qbuf + (size_t)c * 16);
                        accum16<VT, MC>(A, rv, qv);
                    }
                }
                __syncwarp();
                if constexpr (!kFix16) {
                    if (lane == 0 && fetched < total) issue(s);               // may already belong to the next query
                } else {
                    fix_row = rowp;                                           // the stage stays valid until the fix-up below has run
                    fix_stage = s;
                }
            } else {
                const uint8_t *rowp = prm.vec + (size_t)(row0 + r) * prm.pitch;
                if (valid) {
#pragma unroll 4
                    for (int i = 0; i < cnt; ++i) {
                        const int c = p + (i << prm.log2P);
                        const uint4 rv = ldg_stream(reinterpret_cast<const uint4 *>(rowp) + c);
                        const uint4 qv = *reinterpret_cast<const uint4 *>(qbuf + (size_t)c * 16);
                        accum16<VT, MC>(A, rv, qv);
                    }
                }
            }
            accum_reduce(A, P);
            float d = finalize<VT, MC>(A, qn, prm.root);
            if constexpr (kFix16) {
                if (valid && p == 0 && row_needs_exact<VT, MC>(A, qn)) {
                    if constexpr (DIRECT) fix_row = prm.vec + (size_t)(row0 + r) * prm.pitch;
                    d = special_row_distance<VT, MC>(fix_row, qbuf, prm.pitch / 2, prm.root);
                }
                if constexpr (!DIRECT) {
                    __syncwarp();
                    if (lane == 0 && fetched < total) issue(fix_stage);
                }
            }
            if (Q.dist_all != nullptr && valid && p == 0) Q.dist_all[row0 + r] = d;
            if (topk) {
                // rows are visited in scan order (lane order); strict '<' like the reference (:2102, :2145)
                unsigned m = __ballot_sync(0xFFFFFFFFu, valid && p == 0 && d < thr);
                while (m) {
                    const int src = __ffs(m) - 1;
                    m &= m - 1;
                    const float dv = __shfl_sync(0xFFFFFFFFu, d, src);
                    if (dv < thr) {
                        if (lane == 0) {
                            if (logged < prm.logcap) mylog[logged] = make_uint2(__float_as_uint(dv), (uint32_t)(row0 + (src >> prm.log2P)));
                            mylist[pos] = dv;
                        }
                        ++logged;
                        __syncwarp();
                        list_argmax(mylist, prm.kcap, lane, thr, pos);
                    }
                }
            }
        }
        if (topk) {
            __syncwarp();
            if (lane == 0) {
                Q.counts[sidx] = logged;
                if (logged > prm.logcap) atomicExch(&Q.ctrl[1], 1);
            }
            if (prm.kcap == 32) {
                // k <= 32: the CTA's 8 streams are consecutive in scan order.  Sort each stream's list, then one warp merges
                // them in stream order, recording the running k-th value BEFORE each stream (its in-CTA prefix bound), and
                // publishes ONE sorted list per CTA: filter_kernel then walks 148 CTA lists instead of 1184 stream lists.
                float v = (lane < prm.k) ? mylist[lane] : INFINITY;
                v = warp_sort_asc(v, lane);
                mylist[lane] = v;
            } else {
                float *gl = Q.lists + (size_t)sidx * prm.kcap;
                for (int j = lane; j < prm.kcap; j += 32) gl[j] = mylist[j];
            }
        }
        if (g + 1 < prm.nq) {
            // stage the next query into the other buffer: nobody reads that one any more (all warps left query g-1 at its barrier)
            uint4 *dst = reinterpret_cast<uint4 *>(qs + (size_t)((g + 1) & 1) * prm.pitch);
            const uint4 *src = reinterpret_cast<const uint4 *>(prm.q[g + 1].query);
            for (int i = tid; i < prm.nc; i += kThreads) dst[i] = src[i];
        }
        if (g + 1 < prm.nq || (topk && prm.kcap == 32)) __syncthreads();     // query g is complete in this CTA; next query staged
        if (g + 1 == prm.nq && tid == 0 && prm.cta_time != nullptr)
            prm.cta_time[blockIdx.x] = (unsigned)min((long long)0xFFFFFFFFll, (clock64() - clk0) >> 6);   // units of 64 cycles
        if (topk && prm.kcap == 32 && warp == 0) {
            const float *ls = lists_s + (size_t)(g & 1) * kWarps * prm.kcap;
            SortedList Lm;
            Lm.init(lane, prm.k);
            for (int w = 0; w < kWarps; ++w) {
                if (lane == 0) Q.tlocal[(size_t)blockIdx.x * kWarps + w] = Lm.thr;
                Lm.offer_sorted(lane, ls[w * 32 + lane]);
            }
            Q.lists[(size_t)blockIdx.x * 32 + lane] = Lm.v;
        }
    }
}

// ------------------------------------------------------------------ candidate filter
// One warp per stream.  thresholds: a row of stream s can only enter the reference's slots if its distance
// is below the k-th smallest distance among ALL earlier rows; any subset of earlier rows gives a valid upper
// bound.  We use  min( k-th smallest over all streams of earlier segments,
//                      k-th smallest over the earlier streams of the same segment ),
// both built from the streams' final k-lists (each contains the k smallest values of its stream).
//
// Result head of one query, written by filter_kernel and read by the host and by the peers of an exchange:
//   [header: ints kHdr*, kHdrBytes][block table: (first survivor, count) per filter block, kTableCap x int2][survivors]
// Survivors are (distance bits, local row) in scan order once taken block by block through the table; the first
// header[kHdrHeadcap] of them sit in the head, the rest in a separate tail.
constexpr int kHdrTotal = 0;      // survivors of the query
constexpr int kHdrFlags = 1;      // 0, or kHdrOverflow / kHdrLost
constexpr int kHdrSeq = 2;        // launch sequence number of the result slot
constexpr int kHdrBlocks = 3;     // filter blocks: used entries of the block table
constexpr int kHdrXseq = 4;       // exchange sequence number
constexpr int kHdrSrc = 5;        // shard that produced the head
constexpr int kHdrHeadcap = 6;    // survivors carried in the head itself
constexpr int kHdrOverflow = 1;   // flag: the candidate log or the survivor capacity overflowed
constexpr int kHdrLost = 8;       // flag: the receiving side stopped waiting for this head (peer lost)
constexpr int kHdrBytes = 64;     // offset of the block table
constexpr int kTableCap = 512;
constexpr size_t kResHdrBytes = kHdrBytes + sizeof(int2) * kTableCap;   // offset of the survivors

struct FilterQuery {    // per-query pointers of a (group) launch: blockIdx.y selects the query
    const float *lists; // k <= 32: [S / kWarps][32] sorted CTA lists; else [S][kcap] stream lists
    const float *tlocal;// k <= 32: [S] in-CTA prefix bound of each stream (from scan_kernel)
    const uint2 *logs;  // [S][logcap]
    const int *counts;  // [S]
    uint2 *out;         // survivors (dist bits, local row), grouped by block in stream order: the first headcap of them
    uint2 *out_tail;    //   go to out (inside the slot's head, the part that travels), the rest to out_tail
    int2 *table;        // [gridDim.x] (base, count) of each block's survivors in out
    int *hdr;           // the result header (kHdr* fields)
    int *ctrl;          // device: [0] cursor, [1] overflow from scan_kernel, [2] blocks done
    int seqno;
    int xslot;          // push: slot row of the targets' gather buffers
    unsigned xseq;      // push: exchange sequence number published with the head (kHdrXseq) and raised on the flags
};

// NVLink peer-memory all-gather, fused into the filter: the block that completes a query's result head copies the used part
// of it (header, block table, survivors) straight into the gather buffer of every target GPU — peer memory mapped through
// cudaIpc (one process per GPU) or cudaDeviceEnablePeerAccess (one process, several GPUs) — and then raises that target's
// arrival flag with a system-scope release store.  No NCCL kernel, no extra launch, no host synchronisation: the receiving
// side waits on the flags with exchange_wait_kernel on ITS stream and copies the gathered heads to the host.
constexpr int kMaxPeers = 16;
struct PushParams {
    int ntargets;                 // 0: nothing is pushed (single shard)
    int src;                      // this shard's index inside a slot's gather row
    int world;                    // shards per slot in the gather layout [slots][world][head_bytes]
    int head_bytes, res_hdr_bytes;// layout of a head: [header][table][survivors from res_hdr_bytes on]
    int tailcap;                  // survivors beyond the head's headcap travel to a separate tail row of this many entries
    uint8_t *gather[kMaxPeers];   // target t: base of its gather buffer
    unsigned *flags[kMaxPeers];   // target t: [slots][world] arrival flags (the exchange sequence number of the slot)
    uint2 *tails[kMaxPeers];      // target t: [slots][world][tailcap] tail rows (k > 32 on large shards: > headcap survivors)
};

__device__ __forceinline__ void st_release_sys(unsigned *p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// receiving side: one thread per (slot of the group, source shard) spins until that shard's flag carries the expected
// sequence number.  Bounded: after `timeout` clock cycles the missing head is marked (kHdrLost) so that the merge reports
// an error instead of the GPU hanging on a peer that died.
struct WaitParams {
    const unsigned *flags;        // [slots][world]
    uint8_t *gather;              // [slots][world][head_bytes] (local)
    int world, first_slot, nq, head_bytes;
    unsigned xseq[kMaxGroup];
    long long timeout;
};
__global__ void exchange_wait_kernel(const WaitParams wp) {
    const int t = threadIdx.x;
    if (t >= wp.nq * wp.world) return;
    const int j = t / wp.world, r = t % wp.world;
    const size_t at = (size_t)(wp.first_slot + j) * wp.world + r;
    const long long t0 = clock64();
    while (ld_acquire_sys(wp.flags + at) != wp.xseq[j]) {
        if (clock64() - t0 > wp.timeout) {
            reinterpret_cast<int *>(wp.gather + at * wp.head_bytes)[kHdrFlags] = kHdrLost;
            break;
        }
        __nanosleep(200);
    }
}

// the push itself: one block stores the used part of one finished head (header, block table, survivors; the survivors beyond
// headcap from the slot's tail area) into row (xslot, src) of every target and raises the targets' flags.  All threads of the
// block call it; the caller guarantees that the head is complete and visible (filter_kernel: last block; push_heads_kernel:
// stream order after the filters).
__device__ __forceinline__ void push_one_head(const PushParams &pp, const int *hdr, const uint2 *out, const uint2 *out_tail, int xslot, unsigned xseq,
                                              int headcap) {
    const int total = max(__ldcg(hdr + kHdrTotal), 0), nblocks = __ldcg(hdr + kHdrBlocks);
    const int nhead = kHdrBytes / (int)sizeof(uint2) + nblocks;            // uint2 words of header + block table
    const int nsurv = min(total, headcap);
    const int ntail = min(max(total - headcap, 0), pp.tailcap);
    const uint2 *src_head = reinterpret_cast<const uint2 *>(hdr);
    const size_t row = (size_t)xslot * pp.world + pp.src;
    for (int t = 0; t < pp.ntargets; ++t) {
        uint8_t *dst = pp.gather[t] + row * (size_t)pp.head_bytes;
        uint2 *dh = reinterpret_cast<uint2 *>(dst);
        uint2 *ds = reinterpret_cast<uint2 *>(dst + pp.res_hdr_bytes);
        for (int i = (int)threadIdx.x; i < nhead; i += (int)blockDim.x) dh[i] = __ldcg(src_head + i);
        for (int i = (int)threadIdx.x; i < nsurv; i += (int)blockDim.x) ds[i] = __ldcg(out + i);
        if (ntail > 0) {
            uint2 *dt = pp.tails[t] + row * (size_t)pp.tailcap;
            for (int i = (int)threadIdx.x; i < ntail; i += (int)blockDim.x) dt[i] = __ldcg(out_tail + i);
        }
    }
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < pp.ntargets) st_release_sys(pp.flags[threadIdx.x] + row, xseq);
}

// option push_mode = 1: the heads of a finished group are pushed by their own small kernel on the exchange stream instead of by
// the filter's last block (the filter stream then never waits for NVLink acknowledgements)
struct PushGroupParams {
    PushParams push;
    int nq, headcap;
    const int *hdr[kMaxGroup];
    const uint2 *out[kMaxGroup];
    const uint2 *out_tail[kMaxGroup];
    int xslot[kMaxGroup];
    unsigned xseq[kMaxGroup];
};
__global__ void push_heads_kernel(const PushGroupParams gp) {
    const int j = blockIdx.x;
    if (j < gp.nq) push_one_head(gp.push, gp.hdr[j], gp.out[j], gp.out_tail[j], gp.xslot[j], gp.xseq[j], gp.headcap);
}

struct FilterParams {
    PushParams push;
    int S;              // streams
    int k, kcap;
    int logcap;
    int headcap;
    int outcap;         // total capacity (head + tail)
    int nq;             // queries (gridDim.y)
    FilterQuery q[kMaxGroup];
    // adaptive partition (k <= 32 path): the last block turns the scan's per-CTA cycles into new tile bounds, in place
    long long *bounds;          // [ncta + 1] or nullptr
    const unsigned *cta_time;   // [ncta]
    long long total_tiles;
};

constexpr int kFilterWarps = 32;      // generic path: streams (warps) per block
constexpr int kFilterWarpsFast = 8;   // k <= 32 path: small blocks (8 warps, ~21 KB smem) that fit on an SM NEXT TO a scan CTA, so
                                      // that the filter of query i runs while the scan of query i+1 streams (engine: two streams)
__host__ __device__ constexpr int filter_warps(bool fast) { return fast ? kFilterWarpsFast : kFilterWarps; }
// shared memory of the k <= 32 path: [kSegments][32] segment lists | [ncta4] per-CTA bound | [32] segment bounds | [ncta][32] CTA lists
__host__ __device__ constexpr size_t filter_fast_smem(int ncta) {
    return sizeof(float) * ((size_t)8 * 32 + (size_t)((ncta + 3) & ~3) + 32 + (size_t)ncta * 32);
}
constexpr int kSegments = 8;  // threshold segments: few long serial walks beat many short ones (issue-bound otherwise)
constexpr int kLogRegs = 8;   // log entries per lane prefetched into registers (256 per stream)

// FAST: k <= 32: scan_kernel published one sorted list per CTA plus each stream's in-CTA prefix bound; the lists are
// merged in registers (one L2 round trip for 19 KB of lists).
template <bool FAST>
__global__ void __launch_bounds__(filter_warps(FAST) * 32, 1) filter_kernel(const FilterParams fp) {
    constexpr int FW = filter_warps(FAST);
    static_assert(FW >= kSegments, "the segment walks use the first kSegments warps");
    extern __shared__ __align__(16) uint8_t fsm[];
    const FilterQuery &fq = fp.q[blockIdx.y];
    const int k = fp.k, kcap = fp.kcap;
    const int ncta = fp.S / kWarps;                                         // scan CTAs (FAST: each published one sorted list)
    // generic: [32][kcap] segment lists | [32][kcap] scratch | [S] in-segment prefix bound | [32] segment bounds
    // FAST:    see filter_fast_smem (kcap == 32)
    float *seglist = reinterpret_cast<float *>(fsm);
    float *work = seglist + kFilterWarps * kcap;                            // generic only
    float *tlocal = FAST ? seglist + kSegments * 32 : work + kFilterWarps * kcap;   // FAST: per-CTA bound
    float *tseg = tlocal + (FAST ? ((ncta + 3) & ~3) : fp.S);               // [32]
    float *slists = tseg + 32;                                              // FAST: [ncta][32] copy of the CTA lists
    __shared__ int wcount[FW], woff[FW];
    __shared__ int blk_base;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int G = (fp.S + kSegments - 1) / kSegments;                       // streams per segment (generic)

    // ---- issue this warp's log loads first: they do not depend on the thresholds
    const int s = blockIdx.x * FW + warp;
    int n_log = 0;
    uint2 ereg[kLogRegs];
    const uint2 *lg = fq.logs + (size_t)s * fp.logcap;
    if (s < fp.S) n_log = min(fq.counts[s], fp.logcap);
#pragma unroll
    for (int i = 0; i < kLogRegs; ++i) {
        const int j = i * 32 + lane;
        ereg[i] = (j < n_log) ? lg[j] : make_uint2(0x7FC00000u, 0u);       // NaN never survives
    }

    if constexpr (FAST) {
        const int GC = (ncta + kSegments - 1) / kSegments;                  // CTAs per segment
        {   // all CTA lists (ncta x 32 floats, ~19 KB) -> shared memory in one coalesced pass
            const float4 *src = reinterpret_cast<const float4 *>(fq.lists);
            float4 *dst = reinterpret_cast<float4 *>(slists);
            const int tot4 = ncta * 8;
            for (int i = (int)threadIdx.x; i < tot4; i += FW * 32) dst[i] = __ldg(src + i);
        }
        __syncthreads();
        if (warp < kSegments) {   // phase 1: warp g walks the CTAs of segment g in order, recording the running k-th value before each CTA
            SortedList L;
            L.init(lane, k);
            const int c0 = warp * GC, c1 = min(ncta, c0 + GC);
            for (int c = c0; c < c1; ++c) {
                if (lane == 0) tlocal[c] = L.thr;
                L.offer_sorted(lane, slists[c * 32 + lane]);
            }
            seglist[warp * kcap + lane] = L.v;
        }
        __syncthreads();
        if (warp < kSegments) {   // phase 2: warp g merges the lists of segments 0..g-1
            SortedList L;
            L.init(lane, k);
            for (int g = 0; g < warp; ++g) L.offer_sorted(lane, seglist[g * kcap + lane]);
            if (lane == 0) tseg[warp] = L.thr;
        }
        __syncthreads();
    } else {
        // generic path (any k): lists stay in global memory / L2, k-lists in shared memory
        if (warp < kSegments) {
            float *L = seglist + warp * kcap;
            for (int j = lane; j < kcap; j += 32) L[j] = (j < k) ? INFINITY : -INFINITY;
            __syncwarp();
            float thr = INFINITY;
            int pos = 0;
            const int s0 = warp * G, s1 = min(fp.S, s0 + G);
            for (int st = s0; st < s1; ++st) {
                if (lane == 0) tlocal[st] = thr;
                const float *src = fq.lists + (size_t)st * kcap;
                for (int base = 0; base < k; base += 32) {
                    const int j = base + lane;
                    const float v = (j < k) ? src[j] : INFINITY;
                    unsigned m = __ballot_sync(0xFFFFFFFFu, v < thr);
                    while (m) {
                        const int sl = __ffs(m) - 1;
                        m &= m - 1;
                        const float dv = __shfl_sync(0xFFFFFFFFu, v, sl);
                        if (dv < thr) {
                            if (lane == 0) L[pos] = dv;
                            __syncwarp();
                            list_argmax(L, kcap, lane, thr, pos);
                        }
                    }
                }
            }
        }
        __syncthreads();
        if (warp < kSegments) {
            float *L = work + warp * kcap;
            for (int j = lane; j < kcap; j += 32) L[j] = (j < k) ? INFINITY : -INFINITY;
            __syncwarp();
            float thr = INFINITY;
            int pos = 0;
            for (int g = 0; g < warp; ++g) {
                const float *src = seglist + g * kcap;
                for (int base = 0; base < k; base += 32) {
                    const int j = base + lane;
                    const float v = (j < k) ? src[j] : INFINITY;
                    unsigned m = __ballot_sync(0xFFFFFFFFu, v < thr);
                    while (m) {
                        const int sl = __ffs(m) - 1;
                        m &= m - 1;
                        const float dv = __shfl_sync(0xFFFFFFFFu, v, sl);
                        if (dv < thr) {
                            if (lane == 0) L[pos] = dv;
                            __syncwarp();
                            list_argmax(L, kcap, lane, thr, pos);
                        }
                    }
                }
            }
            if (lane == 0) tseg[warp] = thr;
        }
        __syncthreads();
    }

    // ---- phase 3: count, reserve, write — survivors of this block's 32 streams in stream order
    float T = INFINITY;
    if (s < fp.S) {
        if constexpr (FAST) {
            const int c = s / kWarps, GC = (ncta + kSegments - 1) / kSegments;
            T = fminf(fminf(__ldg(fq.tlocal + s), tlocal[c]), tseg[c / GC]);
        } else {
            T = fminf(tlocal[s], tseg[s / G]);
        }
    }
    int mine = 0;
#pragma unroll
    for (int i = 0; i < kLogRegs; ++i) mine += __popc(__ballot_sync(0xFFFFFFFFu, __uint_as_float(ereg[i].x) < T));
    for (int base = kLogRegs * 32; base < n_log; base += 32) {
        const int j = base + lane;
        const bool keep = (j < n_log) && (__uint_as_float(lg[j].x) < T);
        mine += __popc(__ballot_sync(0xFFFFFFFFu, keep));
    }
    if (lane == 0) wcount[warp] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int w = 0; w < FW; ++w) { woff[w] = tot; tot += wcount[w]; }
        const int base = atomicAdd(&fq.ctrl[0], tot);
        blk_base = base;
        fq.table[blockIdx.x] = make_int2(base, tot);
    }
    __syncthreads();
    int wr = blk_base + woff[warp];
#pragma unroll
    for (int i = 0; i < kLogRegs; ++i) {
        const bool keep = __uint_as_float(ereg[i].x) < T;
        const unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
        const int off = wr + __popc(m & ((1u << lane) - 1u));
        if (keep && off < fp.outcap) *(off < fp.headcap ? fq.out + off : fq.out_tail + (off - fp.headcap)) = ereg[i];
        wr += __popc(m);
    }
    for (int base = kLogRegs * 32; base < n_log; base += 32) {
        const int j = base + lane;
        uint2 e = make_uint2(0, 0);
        bool keep = false;
        if (j < n_log) { e = lg[j]; keep = __uint_as_float(e.x) < T; }
        const unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
        const int off = wr + __popc(m & ((1u << lane) - 1u));
        if (keep && off < fp.outcap) *(off < fp.headcap ? fq.out + off : fq.out_tail + (off - fp.headcap)) = e;
        wr += __popc(m);
    }
    if constexpr (FAST) {
        // ---- adaptive partition: share of CTA c for the query after next  ∝  its measured speed (tiles per cycle), damped
        if (fp.bounds != nullptr && blockIdx.x == gridDim.x - 1 && blockIdx.y == gridDim.y - 1 && fp.total_tiles >= 64ll * ncta && ncta <= 1024) {
            __shared__ float spd[1024];
            __shared__ int bad;
            if (threadIdx.x == 0) bad = 0;
            __syncthreads();
            for (int c = threadIdx.x; c < ncta; c += FW * 32) {
                const float tiles = (float)(fp.bounds[c + 1] - fp.bounds[c]);
                const unsigned t = fp.cta_time[c];
                if (t == 0u || !(tiles > 0.0f)) bad = 1;
                spd[c] = tiles / (float)max(t, 1u);
            }
            __syncthreads();
            if (threadIdx.x == 0 && !bad) {
                double sum = 0.0;
                for (int c = 0; c < ncta; ++c) sum += (double)spd[c];
                double acc = 0.0;                       // running boundary in tiles
                long long prev = 0;
                for (int c = 0; c < ncta; ++c) {
                    const double cur = (double)(fp.bounds[c + 1] - prev);            // old share (prev = old bounds[c])
                    const double want = (double)fp.total_tiles * (double)spd[c] / sum;
                    prev = fp.bounds[c + 1];
                    acc += 0.5 * cur + 0.5 * want;
                    long long b = (c == ncta - 1) ? fp.total_tiles : (long long)(acc + 0.5);
                    const long long lo = fp.bounds[c] + kWarps;                       // every CTA keeps at least one tile per warp
                    if (b < lo) b = lo;
                    if (b > fp.total_tiles) b = fp.total_tiles;
                    fp.bounds[c + 1] = b;
                }
            }
            __syncthreads();
        }
    }
    // last block publishes the header and re-arms the control words for the next query.  The host only reads the
    // mapped buffers after the stream has drained, so device-scope ordering between blocks is all that is needed.
    __shared__ int is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const int done = atomicAdd(&fq.ctrl[2], 1);
        const int last = (done == (int)gridDim.x - 1);
        if (last) {
            __threadfence();
            const int total = atomicAdd(&fq.ctrl[0], 0);
            const int ovf = atomicAdd(&fq.ctrl[1], 0);
            fq.hdr[kHdrTotal] = total;
            fq.hdr[kHdrFlags] = (ovf != 0 || total > fp.outcap) ? kHdrOverflow : 0;
            fq.hdr[kHdrSeq] = fq.seqno;
            fq.hdr[kHdrBlocks] = (int)gridDim.x;
            fq.hdr[kHdrXseq] = (int)fq.xseq;
            fq.hdr[kHdrSrc] = fp.push.src;
            fq.hdr[kHdrHeadcap] = fp.headcap;
            fq.ctrl[0] = 0; fq.ctrl[1] = 0; fq.ctrl[2] = 0;
        }
        is_last = last;
    }
    if (fp.push.ntargets > 0) {                                   // uniform across the grid
        __syncthreads();
        if (is_last) {
            // the other blocks' survivors are visible: each fenced before its ctrl[2] increment, thread 0 fenced after
            // observing the last one; read them through L2 (ld.cg), store them to peer memory over NVLink
            push_one_head(fp.push, fq.hdr, fq.out, fq.out_tail, fq.xslot, fq.xseq, fp.headcap);
        }
    }
}

}  // namespace vsb
