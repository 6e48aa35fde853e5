// Device kernels of the batch-exponentiation path, generic over the group descriptor G
// (Bls377G1, Bls377G2, Bw6G1, Bw6G2).  One translation unit per group instantiates them
// (kern_*.cu) and publishes a GroupOps table; api.cu only sees that table.
//
// Data layout in HBM
//   * serialized elements: exactly the reference's byte layout (packed, no header), read/written
//     as u32 words — every element size is a multiple of 16 bytes.
//   * Jacobian scratch `jac`: limb-major SoA, word (c*FW + w) of element i at jac[(c*FW+w)*n + i]
//     (c = X,Y,Z; FW = words per coordinate) so that every warp access is one coalesced 128-byte
//     line.
//   * `prefix`: FW words per element, same limb-major layout, holds the running Z products of the
//     Montgomery batch inversion.
#pragma once
#include <cuda_runtime.h>

#include <cstdlib>
#include <type_traits>

#include "codec.cuh"
#include "glv.cuh"

namespace ss {

// lowest failing index wins: status = min over failures of (index << 8 | code)
constexpr unsigned long long STATUS_OK = ~0ull;

// minimum resident blocks per SM for the 12-limb (G1) instantiations; A/B-measured, see profiles/
#ifndef SS_SUBGROUP_MINB_NARROW
#define SS_SUBGROUP_MINB_NARROW 4
#endif
#ifndef SS_DECODE_MINB_NARROW
#define SS_DECODE_MINB_NARROW 4
#endif

SS_D void report(unsigned long long* status, uint64_t index, int code) {
    atomicMin(status, (unsigned long long)((index << 8) | (uint64_t)code));
}

template <class F>
struct FieldWords;
template <class P>
struct FieldWords<Fp<P>> {
    static constexpr int W = P::N;
    SS_D static void store(uint32_t* base, uint64_t stride, const Fp<P>& a) {
#pragma unroll
        for (int i = 0; i < P::N; i++) base[i * stride] = a.l[i];
    }
    SS_D static Fp<P> load(const uint32_t* base, uint64_t stride) {
        Fp<P> a;
#pragma unroll
        for (int i = 0; i < P::N; i++) a.l[i] = base[i * stride];
        return a;
    }
    SS_D static Fp<P> unpack(const uint32_t* w) {
        Fp<P> a;
#pragma unroll
        for (int i = 0; i < P::N; i++) a.l[i] = w[i];
        return a;
    }
    SS_D static void pack(uint32_t* w, const Fp<P>& a) {
#pragma unroll
        for (int i = 0; i < P::N; i++) w[i] = a.l[i];
    }
};
template <class P>
struct FieldWords<Fp2<P>> {
    static constexpr int W = 2 * P::N;
    SS_D static void store(uint32_t* base, uint64_t stride, const Fp2<P>& a) {
        FieldWords<Fp<P>>::store(base, stride, a.c0);
        FieldWords<Fp<P>>::store(base + P::N * stride, stride, a.c1);
    }
    SS_D static Fp2<P> load(const uint32_t* base, uint64_t stride) {
        Fp2<P> a;
        a.c0 = FieldWords<Fp<P>>::load(base, stride);
        a.c1 = FieldWords<Fp<P>>::load(base + P::N * stride, stride);
        return a;
    }
    SS_D static Fp2<P> unpack(const uint32_t* w) {
        return Fp2<P>{FieldWords<Fp<P>>::unpack(w), FieldWords<Fp<P>>::unpack(w + P::N)};
    }
    SS_D static void pack(uint32_t* w, const Fp2<P>& a) {
        FieldWords<Fp<P>>::pack(w, a.c0);
        FieldWords<Fp<P>>::pack(w + P::N, a.c1);
    }
};

template <class P>
struct FieldWords<Fp3<P>> {
    static constexpr int W = 3 * P::N;
    using B = FieldWords<Fp<P>>;
    SS_D static void store(uint32_t* base, uint64_t stride, const Fp3<P>& a) {
        B::store(base, stride, a.c0);
        B::store(base + P::N * stride, stride, a.c1);
        B::store(base + 2 * P::N * stride, stride, a.c2);
    }
    SS_D static Fp3<P> load(const uint32_t* base, uint64_t stride) {
        return Fp3<P>{B::load(base, stride), B::load(base + P::N * stride, stride), B::load(base + 2 * P::N * stride, stride)};
    }
    SS_D static Fp3<P> unpack(const uint32_t* w) { return Fp3<P>{B::unpack(w), B::unpack(w + P::N), B::unpack(w + 2 * P::N)}; }
    SS_D static void pack(uint32_t* w, const Fp3<P>& a) {
        B::pack(w, a.c0);
        B::pack(w + P::N, a.c1);
        B::pack(w + 2 * P::N, a.c2);
    }
};

// serialized element i of a packed buffer: word-aligned for the ceremony curves, byte-granular for the MNT curves
// (95-byte field elements), see G::BYTE_IO in ec.cuh
template <class G>
SS_D int decode_at(const uint32_t* base, uint64_t i, bool compressed, int check, Affine<typename G::F>& p) {
    const int sz = compressed ? G::CSIZE : G::USIZE;
    if constexpr (G::BYTE_IO) return decode_point<G>(reinterpret_cast<const uint8_t*>(base) + i * sz, compressed, check, p);
    else return decode_point<G>(base + i * (sz / 4), compressed, check, p);
}
template <class G>
SS_D void encode_at(uint32_t* base, uint64_t i, bool compressed, const Affine<typename G::F>& p) {
    const int sz = compressed ? G::CSIZE : G::USIZE;
    if constexpr (G::BYTE_IO) encode_point<G>(reinterpret_cast<uint8_t*>(base) + i * sz, compressed, p);
    else encode_point<G>(base + i * (sz / 4), compressed, p);
}

// ---- scalar preparation -------------------------------------------------------------------------
// tab[j] = tau^(2^j) (Montgomery), j < 64; coeff_m = coeff (Montgomery) or 1.
template <class FrP>
__global__ void k_prepare_scalars(const uint32_t* tau_le, const uint32_t* coeff_le, uint32_t* tab, uint32_t* coeff_m) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    constexpr int N = FrP::N;
    Fp<FrP> t;
    for (int i = 0; i < N; i++) t.l[i] = tau_le[i];
    t = fp_to_mont(t);
    for (int j = 0; j < 64; j++) {
        for (int i = 0; i < N; i++) tab[j * N + i] = t.l[i];
        t = fp_sqr(t);
    }
    Fp<FrP> c = Fp<FrP>::one();
    if (coeff_le) {
        for (int i = 0; i < N; i++) c.l[i] = coeff_le[i];
        c = fp_to_mont(c);
    }
    for (int i = 0; i < N; i++) coeff_m[i] = c.l[i];
}

// tau^e from the table of tau^(2^j)   (== tau.pow([e]), setup-utils/src/helpers.rs:36)
template <class FrP>
SS_D Fp<FrP> tau_power(const uint32_t* __restrict__ tab, uint64_t e) {
    constexpr int N = FrP::N;
    Fp<FrP> r = Fp<FrP>::one();
    bool started = false;
    for (int j = 0; j < 64; j++) {
        if ((e >> j) & 1) {
            Fp<FrP> t;
#pragma unroll
            for (int i = 0; i < N; i++) t.l[i] = __ldg(tab + j * N + i);
            r = started ? fp_mul(r, t) : t;
            started = true;
        }
        if ((e >> j) <= 1) break;
    }
    return r;
}

// generate_powers_of_tau (setup-utils/src/helpers.rs:32-37): out[i] = canonical LE of tau^(start+i)
template <class FrP>
__global__ void k_powers(const uint32_t* __restrict__ tab, uint64_t start, uint64_t n, uint32_t* out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fp<FrP> c = fp_from_mont(tau_power<FrP>(tab, start + i));
#pragma unroll
    for (int k = 0; k < FrP::N; k++) out[i * FrP::N + k] = c.l[k];
}

template <class G>
SS_D void store_affine(uint32_t* aff, uint64_t i, const Affine<typename G::F>& p) {
    using FW = FieldWords<typename G::F>;
    constexpr int W2 = 2 * FW::W;
    uint32_t w[W2];
    FW::pack(w, p.x);
    FW::pack(w + FW::W, p.y);
    uint4* dst = reinterpret_cast<uint4*>(aff + i * W2);
#pragma unroll
    for (int k = 0; k < W2 / 4; k++) dst[k] = make_uint4(w[4 * k], w[4 * k + 1], w[4 * k + 2], w[4 * k + 3]);
}

// Marlin's short scalar vectors (phase1/src/computation.rs:198-257), canonical LE, one thread per degree bound i:
//   dbp_i = tau^(N - 1 - 2^i + 2);  tau_g2[2+i] <- 1/dbp_i;  alpha_g1[3+3i .. 3+3i+3) <- dbp_i * {1, tau, tau^2}
// and the fixed heads tau_g2[0..2) <- {1, tau}, alpha_g1[0..3) <- {1, tau, tau^2} (alpha is applied as `coeff`).
template <class FrP>
__global__ void k_marlin_scalars(const uint32_t* __restrict__ tab, uint64_t powers_length, int k, uint32_t* out_g2,
                                 uint32_t* out_alpha) {
    constexpr int N = FrP::N;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > k) return;
    Fp<FrP> tau, tau2;
#pragma unroll
    for (int w = 0; w < N; w++) {
        tau.l[w] = __ldg(tab + w);
        tau2.l[w] = __ldg(tab + N + w);
    }
    auto put = [&](uint32_t* dst, int slot, const Fp<FrP>& m) {
        Fp<FrP> c = fp_from_mont(m);
#pragma unroll
        for (int w = 0; w < N; w++) dst[slot * N + w] = c.l[w];
    };
    if (i == k) {  // heads
        put(out_g2, 0, Fp<FrP>::one());
        put(out_g2, 1, tau);
        put(out_alpha, 0, Fp<FrP>::one());
        put(out_alpha, 1, tau);
        put(out_alpha, 2, tau2);
        return;
    }
    Fp<FrP> dbp = tau_power<FrP>(tab, powers_length - 1 - (1ull << i) + 2);
    put(out_g2, 2 + i, fp_inv(dbp));
    put(out_alpha, 3 + 3 * i, dbp);
    Fp<FrP> t = fp_mul(dbp, tau);
    put(out_alpha, 3 + 3 * i + 1, t);
    put(out_alpha, 3 + 3 * i + 2, fp_mul(dbp, tau2));
}

// ---- stage 1: read_batch ------------------------------------------------------------------------
// Affine scratch `aff`: [n][2*FW] words (x then y, Montgomery) + one flag byte per element
// (1 = point at infinity).
struct DecodeArgs {
    const uint32_t* in;  // serialized elements
    int in_compressed;
    int check;  // CHECK_*
    uint64_t n;
    uint32_t* aff;
    uint8_t* inf;
    unsigned long long* status;
};

// BatchDeserializer::read_batch (setup-utils/src/io/read.rs:110-135): one element per thread.
template <class G>
__global__ void __launch_bounds__(128, (G::F::CALL_GROUP_OPS ? 1 : SS_DECODE_MINB_NARROW)) k_decode(DecodeArgs a) {
    using F = typename G::F;
    using FW = FieldWords<F>;
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    Affine<F> p;
    int e = decode_at<G>(a.in, i, a.in_compressed != 0, a.check, p);
    if (e != ERR_OK) {
        report(a.status, i, e);
        p.inf = true;
        p.x = F::zero();
        p.y = F::zero();
    }
    store_affine<G>(a.aff, i, p);
    a.inf[i] = p.inf ? 1 : 0;
}

// The affine scratch is ARRAY-OF-STRUCTS: element i = 2*FW contiguous words (x then y), moved with
// 16-byte vector accesses.  Per-element kernels read it as well coalesced as the SoA form would be
// (a warp covers one contiguous 32*8*FW-byte span) and the MSM gathers — random element per lane —
// touch 3 (6) full 32-byte sectors per point instead of 24 (48) partially used ones.
template <class G>
SS_D Affine<typename G::F> load_affine(const uint32_t* aff, const uint8_t* inf, uint64_t /*n*/, uint64_t i) {
    using F = typename G::F;
    using FW = FieldWords<F>;
    constexpr int W2 = 2 * FW::W;
    uint32_t w[W2];
    const uint4* src = reinterpret_cast<const uint4*>(aff + i * W2);
#pragma unroll
    for (int k = 0; k < W2 / 4; k++) {
        uint4 v = src[k];
        w[4 * k] = v.x;
        w[4 * k + 1] = v.y;
        w[4 * k + 2] = v.z;
        w[4 * k + 3] = v.w;
    }
    Affine<F> p;
    p.x = FW::unpack(w);
    p.y = FW::unpack(w + FW::W);
    p.inf = inf[i] != 0;
    return p;
}

// ---- stage 2: batch_exp core --------------------------------------------------------------------
struct ScalarMulArgs {
    const uint32_t* aff;  // decoded bases
    const uint8_t* inf;
    uint64_t n;
    const uint32_t* exps;     // explicit canonical LE scalars [n][FRW], or nullptr
    const uint32_t* tau_tab;  // [64][FRW] Montgomery, used when exps == nullptr
    uint64_t first_power;     // exponent of element 0
    const uint32_t* coeff_m;  // Montgomery coefficient (never null; 1 when absent)
    int has_coeff;
    uint32_t* jac;  // out: Jacobian, limb-major SoA [3*FW][n]
    // group-FFT stages (fft.cuh): the exponent of thread i is first_power + (i & power_mask), and with
    // src_log_m = s >= 0 thread i reads the upper element of butterfly i of a stage with half-size m = 2^s,
    // aff[((i >> s) << (s + 1)) | m | (i & (m - 1))].  Defaults = plain batch_exp.
    // The coefficient is applied to threads i < coeff_limit only (the 1/n of an IFFT rides on block 0's twiddles).
    uint64_t power_mask = ~0ull;
    int src_log_m = -1;
    uint64_t coeff_limit = ~0ull;
    const uint32_t* gather = nullptr;  // sparse dot products (qap.cuh): thread i multiplies aff[gather[i]]
    // fft_compact: the stage skips the butterflies whose twiddle is 1 (j = 0 of every block but block 0, whose
    // twiddle carries the 1/n): thread 0 is (block 0, j 0), thread t >= 1 is block (t-1)/(m-1), j = 1 + (t-1)%(m-1).
    int fft_compact = 0;
    int plain_ladder = 0;  // 1: the reference's double-and-add for inputs that were not subgroup-checked (glv.cuh)
};

// bases[i] <- (exps[i] * coeff?) * bases[i]   (setup-utils/src/helpers.rs:95-106), result left in
// Jacobian form for k_normalize_encode.
#ifndef SS_SMUL_TPB
#define SS_SMUL_TPB 128
#endif
template <class G>
__global__ void __launch_bounds__(SS_SMUL_TPB, G::SMUL_MINB) k_scalar_mul(ScalarMulArgs a) {
    using F = typename G::F;
    using FrP = typename G::Fr::Params;
    using FW = FieldWords<F>;
    constexpr int FRW = FrP::N;
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    uint64_t src = i, pw = i & a.power_mask;
    if (a.src_log_m >= 0) {
        const uint64_t m = 1ull << a.src_log_m;
        uint64_t blk = i >> a.src_log_m, j = i & (m - 1);
        if (a.fft_compact) {
            blk = i ? (i - 1) / (m - 1) : 0;
            j = i ? 1 + (i - 1) % (m - 1) : 0;
            pw = j;
        }
        src = (blk << (a.src_log_m + 1)) | m | j;
    } else if (a.gather) {
        src = a.gather[i];
    }
    Affine<F> base = load_affine<G>(a.aff, a.inf, a.n, src);
    Fp<FrP> s;
    if (a.exps) {
#pragma unroll
        for (int k = 0; k < FRW; k++) s.l[k] = a.exps[i * FRW + k];
        if (a.has_coeff) {
            Fp<FrP> c;
#pragma unroll
            for (int k = 0; k < FRW; k++) c.l[k] = __ldg(a.coeff_m + k);
            s = fp_mul(s, c);  // canonical * Montgomery -> canonical
        }
    } else {
        s = tau_power<FrP>(a.tau_tab, a.first_power + pw);
        if (a.has_coeff && i < a.coeff_limit) {
            Fp<FrP> c;
#pragma unroll
            for (int k = 0; k < FRW; k++) c.l[k] = __ldg(a.coeff_m + k);
            s = fp_mul(s, c);
        }
        s = fp_from_mont(s);
    }
    Jac<F> r;
#if defined(SS_SCALAR_MUL_LADDER)
    r = jac_mul_bits<F>(base, [&](int k) { return s.l[k]; }, FrP::BITS);  // reference algorithm (A/B)
#else
    if constexpr (G::HAS_ENDO) r = scalar_mul_endo<G>(base, s.l, a.plain_ladder != 0);  // GLV / GLS + signed windows + common-Z table (glv.cuh)
    else r = jac_mul_ladder_cold<G>(base, s.l);  // MNT curves: no endomorphism, the reference's double-and-add
#endif
    uint32_t* o = a.jac + i;
    FW::store(o, a.n, r.X);
    FW::store(o + (uint64_t)FW::W * a.n, a.n, r.Y);
    FW::store(o + (uint64_t)2 * FW::W * a.n, a.n, r.Z);
}

// ---- lane-split twins (fp2l.cuh): one element per LANE PAIR, the even lane owns the c0 halves, the odd lane c1 ------
// Same HBM layouts as the per-thread kernels: the affine scratch [n][x.c0 | x.c1 | y.c0 | y.c1] is read as 48-byte
// halves (three 16-byte loads per coordinate), the Jacobian SoA rows (c * FW + 12 * odd + k) are written by the lane
// that owns them.
template <class GL>
SS_D Affine<typename GL::F> load_affine_half(const uint32_t* aff, const uint8_t* inf, uint64_t i) {
    using F = typename GL::F;
    constexpr int HW = F::Base::N;  // words per half coordinate
    const int odd = lane_odd();
    Affine<F> p;
    const uint4* sx = reinterpret_cast<const uint4*>(aff + i * (4 * HW) + odd * HW);
    const uint4* sy = reinterpret_cast<const uint4*>(aff + i * (4 * HW) + 2 * HW + odd * HW);
#pragma unroll
    for (int k = 0; k < HW / 4; k++) {
        const uint4 a = sx[k], b = sy[k];
        p.x.h.l[4 * k] = a.x; p.x.h.l[4 * k + 1] = a.y; p.x.h.l[4 * k + 2] = a.z; p.x.h.l[4 * k + 3] = a.w;
        p.y.h.l[4 * k] = b.x; p.y.h.l[4 * k + 1] = b.y; p.y.h.l[4 * k + 2] = b.z; p.y.h.l[4 * k + 3] = b.w;
    }
    p.inf = inf[i] != 0;
    return p;
}

template <class GL>
__global__ void __launch_bounds__(SS_SMUL_TPB, GL::SMUL_MINB) k_scalar_mul_pair(ScalarMulArgs a) {
    using F = typename GL::F;
    using FrP = typename GL::Fr::Params;
    constexpr int FRW = FrP::N, HW = F::Base::N, FW = 2 * HW;
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = (t >> 1) < a.n;             // both lanes of a pair work on element i
    const uint64_t i = live ? (t >> 1) : a.n - 1;  // out-of-range lanes stay in the warp on a clamped index (fp2l.cuh)
    uint64_t src = i, pw = i & a.power_mask;
    if (a.src_log_m >= 0) {
        const uint64_t m = 1ull << a.src_log_m;
        uint64_t blk = i >> a.src_log_m, j = i & (m - 1);
        if (a.fft_compact) {
            blk = i ? (i - 1) / (m - 1) : 0;
            j = i ? 1 + (i - 1) % (m - 1) : 0;
            pw = j;
        }
        src = (blk << (a.src_log_m + 1)) | m | j;
    } else if (a.gather) {
        src = a.gather[i];
    }
    Affine<F> base = load_affine_half<GL>(a.aff, a.inf, src);
    Fp<FrP> s;  // both lanes derive the same scalar (a few Fr multiplications)
    if (a.exps) {
#pragma unroll
        for (int k = 0; k < FRW; k++) s.l[k] = a.exps[i * FRW + k];
        if (a.has_coeff) {
            Fp<FrP> c;
#pragma unroll
            for (int k = 0; k < FRW; k++) c.l[k] = __ldg(a.coeff_m + k);
            s = fp_mul(s, c);
        }
    } else {
        s = tau_power<FrP>(a.tau_tab, a.first_power + pw);
        if (a.has_coeff && i < a.coeff_limit) {
            Fp<FrP> c;
#pragma unroll
            for (int k = 0; k < FRW; k++) c.l[k] = __ldg(a.coeff_m + k);
            s = fp_mul(s, c);
        }
        s = fp_from_mont(s);
    }
    Jac<F> r = scalar_mul_endo_pair<GL>(base, s.l, a.plain_ladder != 0);
    if (!live) return;
    const int odd = lane_odd();
    uint32_t* o = a.jac + i + (uint64_t)odd * HW * a.n;
#pragma unroll
    for (int k = 0; k < HW; k++) {
        o[(uint64_t)k * a.n] = r.X.h.l[k];
        o[(uint64_t)(FW + k) * a.n] = r.Y.h.l[k];
        o[(uint64_t)(2 * FW + k) * a.n] = r.Z.h.l[k];
    }
}

// ---- stage 3: normalize_batch + write_batch -----------------------------------------------------
struct NormalizeArgs {
    const uint32_t* jac;  // [3*FW][n]
    uint64_t n;
    uint32_t* prefix;  // scratch [FW][n]
    uint32_t* out;     // serialized
    int out_compressed;
    uint32_t threads;  // T: thread t owns elements t, t+T, t+2T, ...
    // when aff_out != nullptr the affine points go to an affine scratch (AoS + flag bytes, as k_decode
    // writes it) instead of being serialized — intermediate stages of the group FFT (fft.cuh)
    uint32_t* aff_out = nullptr;
    uint8_t* inf_out = nullptr;
};

// CurveGroup::normalize_batch (Montgomery's trick, identities skipped) fused with
// BatchSerializer::write_batch (setup-utils/src/helpers.rs:113-114, io/write.rs:57-66).
template <class G>
__global__ void __launch_bounds__(128) k_normalize_encode(NormalizeArgs a) {
    using F = typename G::F;
    using FW = FieldWords<F>;
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.threads || t >= a.n) return;
    const uint64_t n = a.n, T = a.threads;
    const uint32_t* Zb = a.jac + (uint64_t)2 * FW::W * n;
    F acc = F::one();
    uint64_t last = t;
    for (uint64_t e = t; e < n; e += T) {
        F z = FW::load(Zb + e, n);
        if (!z.is_zero()) {
            FW::store(a.prefix + e, n, acc);
            acc = fp_mul(acc, z);
        }
        last = e;
    }
    F inv = fp_inv(acc);
    for (uint64_t e = last;; e -= T) {
        F z = FW::load(Zb + e, n);
        Affine<F> p;
        if (z.is_zero()) {
            p.inf = true;
            p.x = F::zero();
            p.y = F::zero();
        } else {
            F pre = FW::load(a.prefix + e, n);
            F zinv = fp_mul(inv, pre);
            inv = fp_mul(inv, z);
            Jac<F> j;
            j.X = FW::load(a.jac + e, n);
            j.Y = FW::load(a.jac + (uint64_t)FW::W * n + e, n);
            p = jac_to_affine_with_zinv(j, zinv);
        }
        if (a.aff_out) {
            store_affine<G>(a.aff_out, e, p);
            a.inf_out[e] = p.inf ? 1 : 0;
        } else {
            encode_at<G>(a.out, e, a.out_compressed != 0, p);
        }
        if (e < T) break;
    }
}

// ---- write_batch of already-affine elements (decompress / verify re-emit) ------------------------
struct EncodeArgs {
    const uint32_t* aff;
    const uint8_t* inf;
    uint64_t n;  // SoA stride of `aff`
    uint32_t* out;
    int out_compressed;
    uint64_t count;  // elements to encode (<= n)
};

template <class G>
__global__ void __launch_bounds__(128) k_encode(EncodeArgs a) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.count) return;
    Affine<typename G::F> p = load_affine<G>(a.aff, a.inf, a.n, i);
    encode_at<G>(a.out, i, a.out_compressed != 0, p);
}

// ---- p.mul_bigint(r).is_zero() for every element (setup-utils/src/elements.rs:138-142) -----------
struct SubgroupArgs {
    const uint32_t* aff;
    const uint8_t* inf;
    uint64_t n;  // SoA stride of `aff`
    unsigned long long* status;
    uint64_t count;  // elements to check (<= n)
    // 1: the elements were read UNCOMPRESSED without validation, so they need not be on the curve.  The endomorphism
    // tests equal r*P == O only on curve points; the reference runs r*P on whatever it was given
    // (accumulator.rs:120-137), so an off-curve element falls back to that very multiplication (same b-free
    // formulas => same verdict).
    int maybe_off_curve = 0;
};

template <class G>
#if defined(__CUDACC__)
__device__ __noinline__
#endif
bool in_subgroup_rmul_cold(Affine<typename G::F> p) {
    return in_subgroup_rmul<G>(p);
}

template <class G>
__global__ void __launch_bounds__(128, (G::F::CALL_GROUP_OPS ? 1 : SS_SUBGROUP_MINB_NARROW)) k_subgroup(SubgroupArgs a) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.count) return;
    Affine<typename G::F> p = load_affine<G>(a.aff, a.inf, a.n, i);
    bool ok;
    if (a.maybe_off_curve && !on_curve(p, G::b())) ok = in_subgroup_rmul_cold<G>(p);
    else ok = in_subgroup<G>(p);
    if (!ok) report(a.status, i, ERR_INCORRECT_SUBGROUP);
}

// psi(P) == [u] P on the lane-split representation (codec.cuh in_subgroup_endo for Bls377G2), every lane of the warp
// executing the same operations; an infinite element runs on its zero coordinates and is accepted at the end
template <class GL>
SS_D bool in_subgroup_pair(const Affine<typename GL::F>& p, bool maybe_off_curve) {
    using F = typename GL::F;
    using P = typename F::Params;
    Affine<F> q = p;
    q.inf = false;
#if defined(SS_SUBGROUP_RMUL)
    bool ok = jac_mul_bits_pair<P>(q, [](int i) { return GL::GP::order(i); }, GL::GP::ORDER_BITS).Z.is_zero();
#else
    Jac<F> acc{q.x, q.y, F::one()};
#pragma unroll 1
    for (int i = 62; i >= 0; i--) {  // [u] P, u = 0x8508c00000000001 (uniform bits)
        acc = jac_dbl_inl(acc);
        if ((kBls377U >> i) & 1) acc = jac_madd_inl(acc, q);
    }
    F x = q.x, y = q.y;
    Endo<GL>::apply(1, x, y);
    bool ok = jac_eq_affine_pair(acc, x, y);
    // an element read uncompressed without validation may be off the curve: the reference then still runs r * P on its
    // b-free formulas (accumulator.rs:120-137) — reproduce that verdict, warp-wide only when some lane needs it
    if (maybe_off_curve) {
        const bool off = !p.inf && !(fp_sqr(q.y) == fp_add(fp_mul(fp_sqr(q.x), q.x), GL::b()));
        if (warp_any(off)) {
            const bool rm = jac_mul_bits_pair<P>(q, [](int i) { return GL::GP::order(i); }, GL::GP::ORDER_BITS).Z.is_zero();
            ok = off ? rm : ok;
        }
    }
#endif
    return p.inf || ok;
}

template <class GL>
__global__ void __launch_bounds__(128, GL::SMUL_MINB) k_subgroup_pair(SubgroupArgs a) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = (t >> 1) < a.count;
    const uint64_t i = live ? (t >> 1) : a.count - 1;
    Affine<typename GL::F> p = load_affine_half<GL>(a.aff, a.inf, i);
    const bool ok = in_subgroup_pair<GL>(p, a.maybe_off_curve != 0);
    if (live && !ok && !lane_odd()) report(a.status, i, ERR_INCORRECT_SUBGROUP);
}

// ---- sum of a few uncompressed points (adds the per-device partial (s, sx) of a sharded ratio check) ----
template <class G>
__global__ void k_sum_points(const uint32_t* pts, int count, uint32_t* out, unsigned long long* status) {
    using F = typename G::F;
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    Jac<F> acc = Jac<F>::identity();
    for (int i = 0; i < count; i++) {
        Affine<F> p;
        int e = decode_at<G>(pts, (uint64_t)i, false, CHECK_NO, p);
        if (e != ERR_OK) {
            report(status, i, e);
            return;
        }
        acc = jac_madd(acc, p);
    }
    Affine<F> r;
    if (acc.is_identity()) {
        r.inf = true;
        r.x = F::zero();
        r.y = F::zero();
    } else {
        r = jac_to_affine_with_zinv(acc, fp_inv(acc.Z));
    }
    encode_at<G>(out, 0, false, r);
}

// ---- init_element (setup-utils/src/io/write.rs:45-55): the serialized group generator --------------------------
template <class G>
__global__ void k_generator(uint32_t* out, int compressed) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    encode_at<G>(out, 0, compressed != 0, G::generator());
}

// ---- function table seen by api.cu -------------------------------------------------------------
struct GroupOps {
    const char* name;      // e.g. "bls12_377.g1" (profiling labels)
    int usize, csize;      // serialized element sizes
    int fr_words;          // scalar limbs (u32)
    int fr_bytes;          // canonical scalar bytes
    int fr_bits;           // scalar field size in bits
    int has_generator;     // 0: the reference's generator constant of this group is not known (MNT G2)
    int coord_words;       // FW
    void (*prepare_scalars)(const uint32_t* tau_le, const uint32_t* coeff_le, uint32_t* tab, uint32_t* coeff_m,
                            cudaStream_t);
    void (*powers)(const uint32_t* tab, uint64_t start, uint64_t n, uint32_t* out, cudaStream_t);
    void (*marlin_scalars)(const uint32_t* tab, uint64_t powers_length, int k, uint32_t* out_g2, uint32_t* out_alpha, cudaStream_t);
    void (*decode)(const DecodeArgs&, cudaStream_t);
    void (*scalar_mul)(const ScalarMulArgs&, cudaStream_t);
    void (*normalize_encode)(const NormalizeArgs&, cudaStream_t);
    void (*encode)(const EncodeArgs&, cudaStream_t);
    void (*subgroup)(const SubgroupArgs&, cudaStream_t);
    void (*sum_points)(const uint32_t* pts, int count, uint32_t* out, unsigned long long* status, cudaStream_t);
    void (*generator)(uint32_t* out, int compressed, cudaStream_t);
};

template <class G, class = void>
struct HasGenerator : std::true_type {};
template <class G>
struct HasGenerator<G, std::enable_if_t<!G::HAS_GENERATOR>> : std::false_type {};

template <class G>
struct GroupLaunch {
    using FrP = typename G::Fr::Params;
    static void prepare_scalars(const uint32_t* tau_le, const uint32_t* coeff_le, uint32_t* tab, uint32_t* coeff_m,
                                cudaStream_t s) {
        k_prepare_scalars<FrP><<<1, 32, 0, s>>>(tau_le, coeff_le, tab, coeff_m);
    }
    static void powers(const uint32_t* tab, uint64_t start, uint64_t n, uint32_t* out, cudaStream_t s) {
        if (!n) return;
        k_powers<FrP><<<(unsigned)((n + 127) / 128), 128, 0, s>>>(tab, start, n, out);
    }
    static void marlin_scalars(const uint32_t* tab, uint64_t powers_length, int k, uint32_t* out_g2, uint32_t* out_alpha,
                               cudaStream_t s) {
        k_marlin_scalars<FrP><<<(k + 1 + 31) / 32, 32, 0, s>>>(tab, powers_length, k, out_g2, out_alpha);
    }
    // Groups with a lane-split twin (ec.cuh PairTwin): which kernels run it.  $SS_PAIR_KERNELS is a bit mask
    // (1 = scalar multiplication, 2 = subgroup test, 4 = bucket accumulation), default 2: measured on B200 at 2^20
    // (profiles/r02_ab_variants.md) the lane-split subgroup test is 4 % faster than the per-thread one (60.8 vs
    // 63.3 ms: no table, 304-byte frame), the bucket accumulation equal (32.2 vs 32.3 ms) and the scalar multiplication
    // SLOWER (185.6 ms at 255 registers, 207.6 at 168, vs 168.7) — its 8-entry table and the operand exchange keep the
    // per-lane register pressure where the per-thread kernel already was.
    static bool use_pair(int which) {
        static const int mask = [] {
            const char* e = getenv("SS_PAIR_KERNELS");
            return e ? atoi(e) : 2;
        }();
        return (mask & which) != 0;
    }
    static void scalar_mul(const ScalarMulArgs& a, cudaStream_t s) {
        if (!a.n) return;
        using GL = typename PairTwin<G>::type;
        if constexpr (!std::is_void<GL>::value) {
            if (use_pair(1)) {
                k_scalar_mul_pair<GL><<<(unsigned)((2 * a.n + SS_SMUL_TPB - 1) / SS_SMUL_TPB), SS_SMUL_TPB, 0, s>>>(a);
                return;
            }
        }
        k_scalar_mul<G><<<(unsigned)((a.n + SS_SMUL_TPB - 1) / SS_SMUL_TPB), SS_SMUL_TPB, 0, s>>>(a);
    }
    static void normalize_encode(const NormalizeArgs& a, cudaStream_t s) {
        if (!a.n) return;
        k_normalize_encode<G><<<(unsigned)((a.threads + 127) / 128), 128, 0, s>>>(a);
    }
    static void decode(const DecodeArgs& a, cudaStream_t s) {
        if (!a.n) return;
        k_decode<G><<<(unsigned)((a.n + 127) / 128), 128, 0, s>>>(a);
    }
    static void encode(const EncodeArgs& a, cudaStream_t s) {
        if (!a.count) return;
        k_encode<G><<<(unsigned)((a.count + 127) / 128), 128, 0, s>>>(a);
    }
    static void subgroup(const SubgroupArgs& a, cudaStream_t s) {
        if (!a.count) return;
        using GL = typename PairTwin<G>::type;
        if constexpr (!std::is_void<GL>::value) {
            if (use_pair(2)) {
                k_subgroup_pair<GL><<<(unsigned)((2 * a.count + 127) / 128), 128, 0, s>>>(a);
                return;
            }
        }
        k_subgroup<G><<<(unsigned)((a.count + 127) / 128), 128, 0, s>>>(a);
    }
    static void sum_points(const uint32_t* pts, int count, uint32_t* out, unsigned long long* status, cudaStream_t s) {
        k_sum_points<G><<<1, 32, 0, s>>>(pts, count, out, status);
    }
    static void generator(uint32_t* out, int compressed, cudaStream_t s) { k_generator<G><<<1, 32, 0, s>>>(out, compressed); }
    static GroupOps ops() {
        GroupOps o;
        o.name = G::name();
        o.usize = G::USIZE;
        o.csize = G::CSIZE;
        o.fr_words = FrP::N;
        o.fr_bytes = (FrP::BITS + 7) / 8;
        o.fr_bits = FrP::BITS;
        o.has_generator = HasGenerator<G>::value ? 1 : 0;
        o.coord_words = FieldWords<typename G::F>::W;
        o.prepare_scalars = &prepare_scalars;
        o.powers = &powers;
        o.marlin_scalars = &marlin_scalars;
        o.scalar_mul = &scalar_mul;
        o.normalize_encode = &normalize_encode;
        o.decode = &decode;
        o.encode = &encode;
        o.subgroup = &subgroup;
        o.sum_points = &sum_points;
        o.generator = &generator;
        return o;
    }
};

const GroupOps& ops_bls377_g1();
const GroupOps& ops_bls377_g2();
const GroupOps& ops_bw6_g1();
const GroupOps& ops_bw6_g2();
const GroupOps& ops_mnt4_g1();
const GroupOps& ops_mnt4_g2();
const GroupOps& ops_mnt6_g1();
const GroupOps& ops_mnt6_g2();

// out = a^-1 in the scalar field of curve `curve` (ss_curve), Montgomery in and out; kern_fr.cu
void fr_inverse(int curve, const uint32_t* a_mont, uint32_t* out_mont, cudaStream_t s);

}  // namespace ss
