// Random-linear-combination multi-scalar multiplication: merge_pairs / power_pairs
// (setup-utils/src/helpers.rs:371-390) = two `msm_bigint` over the SAME scalars rho_i:
//     s = sum rho_i * v1_i ,  sx = sum rho_i * v2_i          (power_pairs: v2_i = v1_{i+1})
// Pippenger bucket method, one sort shared by both sums:
//   1. k_msm_hist      digit histogram per window                     (atomics on W*B counters)
//   2. k_msm_scan      exclusive scan per window -> bucket offsets
//   3. k_msm_scatter   counting sort of element indices by digit
//   4. k_msm_accumulate one thread per (window, bucket): mixed-adds its run of v1 and v2 points and
//                      folds the result into persistent bucket accumulators (so a vector can be
//                      streamed tile by tile)
//   5. k_msm_reduce1/2/3  running-sum over bucket segments, per-window tree, Horner over windows,
//                      normalise and encode the two results
// The scalars are either supplied (tests, explicit API) or generated on the device from a 256-bit
// seed with ChaCha20 (the reference draws them from thread_rng, helpers.rs:373-376): rho_i is the
// first 128 bits of block i, which keeps the soundness error at 2^-128 while halving the windows.
#pragma once
#include "kernels.cuh"

namespace ss {

// ---- ChaCha20 block function (RFC 8439 quarter rounds; 64-bit block counter, zero nonce) ----------
SS_HD uint32_t rotl32(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }
#define SS_QR(a, b, c, d)                 \
    a += b; d ^= a; d = rotl32(d, 16);    \
    c += d; b ^= c; b = rotl32(b, 12);    \
    a += b; d ^= a; d = rotl32(d, 8);     \
    c += d; b ^= c; b = rotl32(b, 7);

SS_HD void chacha20_block(const uint32_t* key8, uint64_t counter, uint32_t* out16) {
    uint32_t s[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u,
                      key8[0], key8[1], key8[2], key8[3], key8[4], key8[5], key8[6], key8[7],
                      (uint32_t)counter, (uint32_t)(counter >> 32), 0u, 0u};
    uint32_t x[16];
#pragma unroll
    for (int i = 0; i < 16; i++) x[i] = s[i];
#pragma unroll 1
    for (int r = 0; r < 10; r++) {
        SS_QR(x[0], x[4], x[8], x[12]) SS_QR(x[1], x[5], x[9], x[13]) SS_QR(x[2], x[6], x[10], x[14]) SS_QR(x[3], x[7], x[11], x[15])
        SS_QR(x[0], x[5], x[10], x[15]) SS_QR(x[1], x[6], x[11], x[12]) SS_QR(x[2], x[7], x[8], x[13]) SS_QR(x[3], x[4], x[9], x[14])
    }
#pragma unroll
    for (int i = 0; i < 16; i++) out16[i] = x[i] + s[i];
}
#undef SS_QR

struct RhoSource {
    const uint32_t* explicit_rho;  // [n][frw] canonical LE, or nullptr
    uint32_t key[8];               // ChaCha20 key when explicit_rho == nullptr
    uint64_t first_index;          // global index of element 0 (ChaCha counter base)
    int frw;                       // scalar words
    int nbits;                     // scalar bits actually used (128 = W*c for generated, field bits for explicit)
};

// c-bit digit `w` of the scalar of element i
SS_D uint32_t rho_digit(const RhoSource& r, const uint32_t* words, int w, int c) {
    const int bit = w * c;
    if (bit >= r.nbits) return 0;
    const int lo = bit >> 5, sh = bit & 31;
    uint64_t v = words[lo];
    if (lo + 1 < r.frw && sh + c > 32) v |= (uint64_t)words[lo + 1] << 32;
    uint32_t d = (uint32_t)(v >> sh) & ((1u << c) - 1);
    const int left = r.nbits - bit;
    if (left < c) d &= (1u << left) - 1;
    return d;
}

SS_D void rho_load(const RhoSource& r, uint64_t i, uint32_t* words /*[24]*/) {
    if (r.explicit_rho) {
        for (int k = 0; k < r.frw; k++) words[k] = r.explicit_rho[i * r.frw + k];
    } else {
        uint32_t blk[16];
        chacha20_block(r.key, r.first_index + i, blk);
        for (int k = 0; k < r.frw; k++) words[k] = k < 5 ? blk[k] : 0u;  // up to 160 bits; nbits masks the rest
    }
}

struct MsmSortArgs {
    RhoSource rho;
    uint64_t n;   // pairs in this tile
    int c, W;     // window bits, windows
    uint32_t* hist;    // [W][B]   counts, then (after scan) exclusive offsets
    uint32_t* cursor;  // [W][B]
    uint32_t* idx;     // [W][n]
};

static __global__ void k_msm_hist(MsmSortArgs a) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    uint32_t words[24];
    rho_load(a.rho, i, words);
    const uint32_t B = 1u << a.c;
    for (int w = 0; w < a.W; w++) {
        uint32_t d = rho_digit(a.rho, words, w, a.c);
        if (d) atomicAdd(&a.hist[(size_t)w * B + d], 1u);
    }
}

// one block per window: exclusive scan of B counters (B <= 2^16), writes offsets to hist and cursor
static __global__ void k_msm_scan(uint32_t* hist, uint32_t* cursor, uint32_t* counts, int c) {
    const uint32_t B = 1u << c;
    uint32_t* h = hist + (size_t)blockIdx.x * B;
    uint32_t* cu = cursor + (size_t)blockIdx.x * B;
    uint32_t* cn = counts + (size_t)blockIdx.x * B;
    __shared__ uint32_t part[1024];
    const uint32_t per = (B + blockDim.x - 1) / blockDim.x;
    const uint32_t lo = threadIdx.x * per, hi = min(B, lo + per);
    uint32_t s = 0;
    for (uint32_t k = lo; k < hi; k++) s += h[k];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (uint32_t t = 0; t < blockDim.x; t++) {
            uint32_t v = part[t];
            part[t] = run;
            run += v;
        }
    }
    __syncthreads();
    uint32_t run = part[threadIdx.x];
    for (uint32_t k = lo; k < hi; k++) {
        uint32_t v = h[k];
        cn[k] = v;
        h[k] = run;
        cu[k] = run;
        run += v;
    }
}

static __global__ void k_msm_scatter(MsmSortArgs a) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    uint32_t words[24];
    rho_load(a.rho, i, words);
    const uint32_t B = 1u << a.c;
    for (int w = 0; w < a.W; w++) {
        uint32_t d = rho_digit(a.rho, words, w, a.c);
        if (d) {
            uint32_t pos = atomicAdd(&a.cursor[(size_t)w * B + d], 1u);
            a.idx[(size_t)w * a.n + pos] = (uint32_t)i;
        }
    }
}

// ---- bucket accumulators ------------------------------------------------------------------------
// Layout: [NB][3*FW] with NB = 2 * W * B  (first W*B entries: sums over v1, second: over v2).
// Bucket / partial-sum arrays are ARRAY-OF-STRUCTS: entry i = 3*FW contiguous words (X, Y, Z), moved
// with 16-byte vector accesses.  (The limb-major SoA form used elsewhere puts the 3*FW words of one
// bucket 2*W*B*4 bytes apart; with buckets visited in sorted-by-run-length order that is 36 scattered
// sectors per bucket and, for some power-of-two strides, pathological: 3.2 s instead of 9 ms for a
// 2^19-element vector, profiles/r01_ab_variants.md.)  `stride` is kept in the signature for symmetry.
template <class G>
SS_D Jac<typename G::F> load_jac(const uint32_t* base, uint64_t /*stride*/, uint64_t i) {
    using FW = FieldWords<typename G::F>;
    constexpr int W3 = 3 * FW::W;
    uint32_t w[W3];
    const uint4* src = reinterpret_cast<const uint4*>(base + i * W3);
#pragma unroll
    for (int k = 0; k < W3 / 4; k++) {
        uint4 v = src[k];
        w[4 * k] = v.x;
        w[4 * k + 1] = v.y;
        w[4 * k + 2] = v.z;
        w[4 * k + 3] = v.w;
    }
    Jac<typename G::F> j;
    j.X = FW::unpack(w);
    j.Y = FW::unpack(w + FW::W);
    j.Z = FW::unpack(w + 2 * FW::W);
    return j;
}
template <class G>
SS_D void store_jac(uint32_t* base, uint64_t /*stride*/, uint64_t i, const Jac<typename G::F>& j) {
    using FW = FieldWords<typename G::F>;
    constexpr int W3 = 3 * FW::W;
    uint32_t w[W3];
    FW::pack(w, j.X);
    FW::pack(w + FW::W, j.Y);
    FW::pack(w + 2 * FW::W, j.Z);
    uint4* dst = reinterpret_cast<uint4*>(base + i * W3);
#pragma unroll
    for (int k = 0; k < W3 / 4; k++) dst[k] = make_uint4(w[4 * k], w[4 * k + 1], w[4 * k + 2], w[4 * k + 3]);
}

template <class G>
__global__ void k_jac_fill_identity(uint32_t* base, uint64_t count) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    store_jac<G>(base, count, i, Jac<typename G::F>::identity());
}

struct MsmAccArgs {
    const uint32_t* aff1;  // SoA stride `stride`
    const uint8_t* inf1;
    const uint32_t* aff2;
    const uint8_t* inf2;
    uint64_t stride;
    uint64_t n;  // pairs in this tile
    int c, W;
    const uint32_t* offsets;  // [W][B] exclusive offsets
    const uint32_t* counts;   // [W][B]
    const uint32_t* idx;      // [W][n]
    const uint32_t* order;    // [W*B] bucket ids sorted by decreasing run length
    uint32_t* buckets;        // [3*FW][2*W*B]
};

#ifndef SS_MSM_MINB_NARROW
#define SS_MSM_MINB_NARROW 3
#endif
template <class G>
__global__ void __launch_bounds__(128, (G::F::CALL_GROUP_OPS ? 1 : SS_MSM_MINB_NARROW)) k_msm_accumulate(MsmAccArgs a) {
    using F = typename G::F;
    const uint32_t B = 1u << a.c;
    const uint64_t WB = (uint64_t)a.W * B;
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= WB) return;
    // buckets are visited longest-run first: the lanes of a warp get runs of (nearly) equal length and the
    // tail of the grid is made of the short ones
    const uint64_t t = a.order[tid];
    const uint32_t d = (uint32_t)(t & (B - 1));
    const uint32_t cnt = a.counts[t];
    if (d == 0 || cnt == 0) return;
    const int w = (int)(t >> a.c);
    const uint32_t* list = a.idx + (size_t)w * a.n + a.offsets[t];
    Jac<F> s1 = Jac<F>::identity(), s2 = Jac<F>::identity();
    for (uint32_t k = 0; k < cnt; k++) {
        const uint32_t i = list[k];
        s1 = jac_madd(s1, load_affine<G>(a.aff1, a.inf1, a.stride, i));
        s2 = jac_madd(s2, load_affine<G>(a.aff2, a.inf2, a.stride, i));
    }
    const uint64_t NB = 2 * WB;
    store_jac<G>(a.buckets, NB, t, jac_add(load_jac<G>(a.buckets, NB, t), s1));
    store_jac<G>(a.buckets, NB, WB + t, jac_add(load_jac<G>(a.buckets, NB, WB + t), s2));
}

// lane-split twin: one bucket per lane pair (fp2l.cuh); bucket entries are read / written as their 48-byte halves
template <class GL>
SS_D Jac<typename GL::F> load_jac_half(const uint32_t* base, uint64_t i) {
    using F = typename GL::F;
    constexpr int HW = F::Base::N;
    const int odd = lane_odd();
    Jac<F> j;
    const uint4* s = reinterpret_cast<const uint4*>(base + i * (6 * HW) + odd * HW);
#pragma unroll
    for (int k = 0; k < HW / 4; k++) {
        const uint4 a = s[k], b = s[k + 2 * HW / 4], c = s[k + 4 * HW / 4];
        j.X.h.l[4 * k] = a.x; j.X.h.l[4 * k + 1] = a.y; j.X.h.l[4 * k + 2] = a.z; j.X.h.l[4 * k + 3] = a.w;
        j.Y.h.l[4 * k] = b.x; j.Y.h.l[4 * k + 1] = b.y; j.Y.h.l[4 * k + 2] = b.z; j.Y.h.l[4 * k + 3] = b.w;
        j.Z.h.l[4 * k] = c.x; j.Z.h.l[4 * k + 1] = c.y; j.Z.h.l[4 * k + 2] = c.z; j.Z.h.l[4 * k + 3] = c.w;
    }
    return j;
}
template <class GL>
SS_D void store_jac_half(uint32_t* base, uint64_t i, const Jac<typename GL::F>& j) {
    using F = typename GL::F;
    constexpr int HW = F::Base::N;
    const int odd = lane_odd();
    uint4* d = reinterpret_cast<uint4*>(base + i * (6 * HW) + odd * HW);
#pragma unroll
    for (int k = 0; k < HW / 4; k++) {
        d[k] = make_uint4(j.X.h.l[4 * k], j.X.h.l[4 * k + 1], j.X.h.l[4 * k + 2], j.X.h.l[4 * k + 3]);
        d[k + 2 * HW / 4] = make_uint4(j.Y.h.l[4 * k], j.Y.h.l[4 * k + 1], j.Y.h.l[4 * k + 2], j.Y.h.l[4 * k + 3]);
        d[k + 4 * HW / 4] = make_uint4(j.Z.h.l[4 * k], j.Z.h.l[4 * k + 1], j.Z.h.l[4 * k + 2], j.Z.h.l[4 * k + 3]);
    }
}

template <class GL>
__global__ void __launch_bounds__(128, GL::SMUL_MINB) k_msm_accumulate_pair(MsmAccArgs a) {
    using F = typename GL::F;
    const uint32_t B = 1u << a.c;
    const uint64_t WB = (uint64_t)a.W * B;
    const uint64_t tid = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    // converged-warp discipline (fp2l.cuh): no lane leaves early; a warp walks max(run length) steps — buckets are
    // visited in order of decreasing run length, so the runs of one warp are (nearly) equal — and lanes whose run is
    // over add the point at infinity
    const bool valid = tid < WB;
    const uint64_t t = valid ? a.order[tid] : 0;
    const uint32_t d = (uint32_t)(t & (B - 1));
    const bool active = valid && d != 0 && a.counts[t] != 0;
    const uint32_t cnt = active ? a.counts[t] : 0u;
    const int w = (int)(t >> a.c);
    const uint32_t* list = a.idx + (size_t)w * a.n + (active ? a.offsets[t] : 0u);
    const uint32_t steps = __reduce_max_sync(kFullMask, cnt);
    Jac<F> s1 = Jac<F>::identity(), s2 = Jac<F>::identity();
#pragma unroll 1
    for (uint32_t k = 0; k < steps; k++) {
        const bool on = k < cnt;
        const uint32_t i = on ? list[k] : 0u;
        Affine<F> q1 = load_affine_half<GL>(a.aff1, a.inf1, i);
        Affine<F> q2 = load_affine_half<GL>(a.aff2, a.inf2, i);
        q1.inf = q1.inf || !on;
        q2.inf = q2.inf || !on;
        s1 = jac_madd_inl(s1, q1);
        s2 = jac_madd_inl(s2, q2);
    }
    const Jac<F> b1 = jac_add_inl(load_jac_half<GL>(a.buckets, t), s1);
    const Jac<F> b2 = jac_add_inl(load_jac_half<GL>(a.buckets, WB + t), s2);
    if (active) {
        store_jac_half<GL>(a.buckets, t, b1);
        store_jac_half<GL>(a.buckets, WB + t, b2);
    }
}

// k * P for a small k (Jacobian base)
template <class F>
SS_D Jac<F> jac_mul_small(const Jac<F>& p, uint32_t k) {
    if (k == 0) return Jac<F>::identity();
    // start below the leading bit: a serial tail kernel pays for every doubling, also those of the identity
    Jac<F> acc = p;
    for (int b = 30 - __clz(k); b >= 0; b--) {
        acc = jac_dbl(acc);
        if ((k >> b) & 1) acc = jac_add(acc, p);
    }
    return acc;
}

struct MsmReduceArgs {
    const uint32_t* buckets;  // [3*FW][2*W*B]
    int c, W;
    uint32_t seglen, nseg;  // B = seglen * nseg
    uint32_t* segres;       // [3*FW][2*W*nseg]
    uint32_t* winres;       // [3*FW][2*W]
    uint32_t* out_s;        // uncompressed encodings
    uint32_t* out_sx;
};

// one thread per (sum, window, segment): sum_{d in seg} d * B_d
template <class G>
__global__ void __launch_bounds__(128) k_msm_reduce1(MsmReduceArgs a) {
    using F = typename G::F;
    const uint32_t B = 1u << a.c;
    const uint64_t total = (uint64_t)2 * a.W * a.nseg;
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const uint32_t seg = (uint32_t)(t % a.nseg);
    const uint64_t sw = t / a.nseg;  // sum * W + window
    const uint64_t NB = (uint64_t)2 * a.W * B;
    const uint32_t lo = seg * a.seglen, hi = lo + a.seglen;
    Jac<F> run = Jac<F>::identity(), acc = Jac<F>::identity();
    for (uint32_t d = hi; d-- > lo;) {
        run = jac_add(run, load_jac<G>(a.buckets, NB, sw * B + d));
        acc = jac_add(acc, run);
    }
    // acc = sum (d - lo + 1) B_d ; want sum d B_d = acc + (lo - 1) * run   (lo = 0: acc - run)
    Jac<F> r;
    if (lo == 0) {
        Jac<F> nr = run;
        nr.Y = fp_neg(nr.Y);
        r = jac_add(acc, nr);
    } else {
        r = jac_add(acc, jac_mul_small(run, lo - 1));
    }
    store_jac<G>(a.segres, total, t, r);
}

// grid (W, 2), REDUCE2_THREADS<F> threads: every thread sums a slice of the window's segment results, then a
// shared-memory tree (log2 T dependent additions instead of the T - 1 a single finishing thread would chain)
template <class F>
struct Reduce2Threads {
    static constexpr int value = sizeof(Jac<F>) * 128 <= 40960 ? 128 : (sizeof(Jac<F>) * 64 <= 40960 ? 64 : 32);
};
template <class G>
__global__ void k_msm_reduce2(MsmReduceArgs a) {
    using F = typename G::F;
    constexpr int T = Reduce2Threads<F>::value;
    __shared__ Jac<F> part[T];
    const uint64_t sw = (uint64_t)blockIdx.y * a.W + blockIdx.x;
    const uint64_t total = (uint64_t)2 * a.W * a.nseg;
    Jac<F> s = Jac<F>::identity();
    for (uint32_t k = threadIdx.x; k < a.nseg; k += T) s = jac_add(s, load_jac<G>(a.segres, total, sw * a.nseg + k));
    part[threadIdx.x] = s;
    __syncthreads();
    for (int h = T / 2; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) part[threadIdx.x] = jac_add(part[threadIdx.x], part[threadIdx.x + h]);
        __syncthreads();
    }
    if (threadIdx.x == 0) store_jac<G>(a.winres, (uint64_t)2 * a.W, sw, part[0]);
}

// 2 threads: Horner over windows, normalise, encode uncompressed
template <class G>
__global__ void k_msm_reduce3(MsmReduceArgs a) {
    using F = typename G::F;
    const int which = threadIdx.x;
    if (which > 1 || blockIdx.x != 0) return;
    Jac<F> r = load_jac<G>(a.winres, (uint64_t)2 * a.W, (uint64_t)which * a.W + a.W - 1);
    for (int w = a.W - 2; w >= 0; w--) {
        for (int k = 0; k < a.c; k++) r = jac_dbl(r);
        r = jac_add(r, load_jac<G>(a.winres, (uint64_t)2 * a.W, (uint64_t)which * a.W + w));
    }
    Affine<F> p;
    if (r.is_identity()) {
        p.inf = true;
        p.x = F::zero();
        p.y = F::zero();
    } else {
        p = jac_to_affine_with_zinv(r, fp_inv(r.Z));
    }
    encode_at<G>(which == 0 ? a.out_s : a.out_sx, 0, false, p);
}

// ---- launchers ----------------------------------------------------------------------------------
struct MsmOps {
    void (*fill_identity)(uint32_t* base, uint64_t count, cudaStream_t);
    void (*accumulate)(const MsmAccArgs&, cudaStream_t);
    void (*reduce)(const MsmReduceArgs&, cudaStream_t);
};

template <class G>
struct MsmLaunch {
    static void fill_identity(uint32_t* base, uint64_t count, cudaStream_t s) {
        k_jac_fill_identity<G><<<(unsigned)((count + 255) / 256), 256, 0, s>>>(base, count);
    }
    static void accumulate(const MsmAccArgs& a, cudaStream_t s) {
        const uint64_t wb = (uint64_t)a.W << a.c;
        using GL = typename PairTwin<G>::type;
        if constexpr (!std::is_void<GL>::value) {
            if (GroupLaunch<G>::use_pair(4)) {
                k_msm_accumulate_pair<GL><<<(unsigned)((2 * wb + 127) / 128), 128, 0, s>>>(a);
                return;
            }
        }
        k_msm_accumulate<G><<<(unsigned)((wb + 127) / 128), 128, 0, s>>>(a);
    }
    static void reduce(const MsmReduceArgs& a, cudaStream_t s) {
        const uint64_t t1 = (uint64_t)2 * a.W * a.nseg;
        k_msm_reduce1<G><<<(unsigned)((t1 + 127) / 128), 128, 0, s>>>(a);
        k_msm_reduce2<G><<<dim3(a.W, 2), Reduce2Threads<typename G::F>::value, 0, s>>>(a);
        k_msm_reduce3<G><<<1, 32, 0, s>>>(a);
    }
    static MsmOps ops() { return MsmOps{&fill_identity, &accumulate, &reduce}; }
};

// counting sort of the W*B buckets by decreasing run length (runs longer than 255 share the first bin)
static __global__ void k_msm_order_hist(const uint32_t* counts, uint64_t wb, uint32_t* bins) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= wb) return;
    uint32_t c = counts[t];
    atomicAdd(&bins[255u - (c > 255u ? 255u : c)], 1u);
}
static __global__ void k_msm_order_scan(uint32_t* bins) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t run = 0;
    for (int i = 0; i < 256; i++) {
        uint32_t v = bins[i];
        bins[i] = run;
        run += v;
    }
}
static __global__ void k_msm_order_scatter(const uint32_t* counts, uint64_t wb, uint32_t* bins, uint32_t* order) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= wb) return;
    uint32_t c = counts[t];
    uint32_t pos = atomicAdd(&bins[255u - (c > 255u ? 255u : c)], 1u);
    order[pos] = (uint32_t)t;
}

static inline void msm_order(const uint32_t* counts, uint64_t wb, uint32_t* bins, uint32_t* order, cudaStream_t s) {
    cudaMemsetAsync(bins, 0, 256 * 4, s);
    k_msm_order_hist<<<(unsigned)((wb + 255) / 256), 256, 0, s>>>(counts, wb, bins);
    k_msm_order_scan<<<1, 32, 0, s>>>(bins);
    k_msm_order_scatter<<<(unsigned)((wb + 255) / 256), 256, 0, s>>>(counts, wb, bins, order);
}

static inline void msm_sort(const MsmSortArgs& a, uint32_t* counts, cudaStream_t s) {
    const uint32_t B = 1u << a.c;
    cudaMemsetAsync(a.hist, 0, (size_t)a.W * B * 4, s);
    k_msm_hist<<<(unsigned)((a.n + 255) / 256), 256, 0, s>>>(a);
    k_msm_scan<<<a.W, B < 1024 ? B : 1024, 0, s>>>(a.hist, a.cursor, counts, a.c);
    k_msm_scatter<<<(unsigned)((a.n + 255) / 256), 256, 0, s>>>(a);
}

const MsmOps& msm_ops_bls377_g1();
const MsmOps& msm_ops_bls377_g2();
const MsmOps& msm_ops_bw6_g1();
const MsmOps& msm_ops_bw6_g2();
const MsmOps& msm_ops_mnt4_g1();
const MsmOps& msm_ops_mnt4_g2();
const MsmOps& msm_ops_mnt6_g1();
const MsmOps& msm_ops_mnt6_g2();

}  // namespace ss
