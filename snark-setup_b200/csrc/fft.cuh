// Group inverse FFT over curve points and the Groth16 H query — the device side of
// Groth16Params::new (setup-utils/src/groth16_utils.rs:44-63,81-131; SURVEY.md §8f rank 3):
//
//   to_coeffs:   coeffs_j = (1/n) * sum_i  w^(-i*j) * P_i      (domain.ifft over C::Group, then normalize_batch)
//   h_query:     h_i      = P_(i+m) - P_i,  i < m - 1           (groth16_utils.rs:59-63)
//
// The result of an IFFT is a mathematical object (w = the domain's group_gen is fixed by ark-ff/ark-poly,
// see FrP::fft_root), and the outputs cross the boundary as canonical affine bytes, so any exact algorithm
// is bit-identical to arkworks' in_order_ifft_in_place.  Here: radix-2 decimation in time.
//   1. bit-reversal gather of the decoded points                                  k_fft_bitrev   (HBM-bound)
//   2. stage s = 0 .. log n - 1 (half-size m = 2^s, w_s = w^(-n/2m)):
//        t_i  = w_s^(i mod m) * upper_i      k_scalar_mul on the gathered upper elements whose twiddle is not 1
//                                            (none for s = 0; j = 0 of every block but block 0 is skipped)
//        lo', hi' = lo + t, lo - t           k_fft_butterfly, two mixed additions (exceptional cases handled)
//        batch-normalise to affine           k_normalize_encode -> affine scratch (last stage: serialized bytes)
//   The final scaling by n^-1 costs no scalar multiplications of its own: block 0 of every stage uses the
//   twiddles n^-1 * w_s^j (its lower half is block 0 of the previous stage, already scaled), and only
//   elements 0 and 1 are multiplied by n^-1 directly before the twiddle-free stage 0.
// Twiddle scalars are never materialised: thread i derives w_s^(i mod m) from the table of w_s^(2^j), which for
// every stage is a window of ONE sequence seq[j] = (w^-1)^(2^j) (w_s^(2^j) = seq[log n - 1 - s + j]).
// Work: about (log n - 2) * n/2 scalar multiplications — the integer-multiply pipe bounds it like batch_exp.
#pragma once
#include "kernels.cuh"

namespace ss {

// seq[j] = (w_n^-1)^(2^j) for j < log_n + 64 (Montgomery; 1 from j = log_n on), ninv_m = n^-1 (Montgomery).
template <class FrP>
__global__ void k_fft_prepare(int log_n, uint32_t* seq, uint32_t* ninv_m) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    constexpr int N = FrP::N;
    Fp<FrP> w;
    for (int i = 0; i < N; i++) w.l[i] = FrP::fft_root(i);
    // F::get_root_of_unity (ark-ff fields/mod.rs): square TWO_ADIC_ROOT_OF_UNITY down to order 2^log_n
    for (int i = log_n; i < FrP::TWO_ADICITY; i++) w = fp_sqr(w);
    w = fp_inv(w);
    for (int j = 0; j < log_n + 64; j++) {
        for (int i = 0; i < N; i++) seq[j * N + i] = w.l[i];
        w = fp_sqr(w);
    }
    Fp<FrP> nn = Fp<FrP>::zero();
    nn.l[log_n >> 5] = 1u << (log_n & 31);
    nn = fp_inv(fp_to_mont(nn));
    for (int i = 0; i < N; i++) ninv_m[i] = nn.l[i];
}

static __device__ __forceinline__ uint64_t bit_reverse(uint64_t v, int bits) { return bits ? (__brevll(v) >> (64 - bits)) : 0; }

// dst[i] = src[bitrev(i)]; affine scratch is AoS of 2*FW words, moved as 16-byte vectors
template <class G>
__global__ void k_fft_bitrev(const uint32_t* __restrict__ src, const uint8_t* __restrict__ src_inf, uint32_t* dst,
                             uint8_t* dst_inf, int log_n) {
    constexpr int V = 2 * FieldWords<typename G::F>::W / 4;  // uint4 per element
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t e = t / V, k = t % V;
    if (e >> log_n) return;
    const uint64_t r = bit_reverse(e, log_n);
    reinterpret_cast<uint4*>(dst)[e * V + k] = reinterpret_cast<const uint4*>(src)[r * V + k];
    if (k == 0) dst_inf[e] = src_inf[r];
}

template <class G>
SS_D Jac<typename G::F> load_jac_soa(const uint32_t* jac, uint64_t stride, uint64_t i) {
    using FW = FieldWords<typename G::F>;
    Jac<typename G::F> r;
    r.X = FW::load(jac + i, stride);
    r.Y = FW::load(jac + (uint64_t)FW::W * stride + i, stride);
    r.Z = FW::load(jac + (uint64_t)2 * FW::W * stride + i, stride);
    return r;
}
template <class G>
SS_D void store_jac_soa(uint32_t* jac, uint64_t stride, uint64_t i, const Jac<typename G::F>& p) {
    using FW = FieldWords<typename G::F>;
    FW::store(jac + i, stride, p.X);
    FW::store(jac + (uint64_t)FW::W * stride + i, stride, p.Y);
    FW::store(jac + (uint64_t)2 * FW::W * stride + i, stride, p.Z);
}

struct ButterflyArgs {
    const uint32_t* aff;  // n affine points (stage input)
    const uint8_t* inf;
    const uint32_t* tw;  // twiddled upper halves, Jacobian SoA [3*FW][tw_count], or nullptr (twiddle 1: read aff)
    uint64_t n;          // power of two >= 2
    int log_m;           // stage: half-size m = 2^log_m
    uint32_t* jac;       // out: Jacobian SoA [3*FW][n], natural positions
    // compact twiddle array (ScalarMulArgs::fft_compact): entry 0 = (block 0, j 0), entry 1 + blk (m-1) + (j-1) for
    // j >= 1; the j = 0 butterflies of the other blocks have twiddle 1 and read their upper element from `aff`
    uint64_t tw_count;
    int compact;
};

// butterfly i: lo = ((i >> s) << (s+1)) | (i & (m-1)), hi = lo | m;  (lo, hi) <- (lo + t, lo - t)
template <class G>
__global__ void __launch_bounds__(128) k_fft_butterfly(ButterflyArgs a) {
    using F = typename G::F;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t half = a.n >> 1;
    if (i >= half) return;
    const uint64_t m = 1ull << a.log_m;
    const uint64_t lo = ((i >> a.log_m) << (a.log_m + 1)) | (i & (m - 1)), hi = lo | m;
    Affine<F> u = load_affine<G>(a.aff, a.inf, a.n, lo);
    Jac<F> t;
    const uint64_t blk = i >> a.log_m, j = i & (m - 1);
    if (a.tw && !(a.compact && j == 0 && blk != 0)) {
        const uint64_t ti = a.compact ? (j == 0 ? 0 : 1 + blk * (m - 1) + (j - 1)) : i;
        t = load_jac_soa<G>(a.tw, a.tw_count, ti);
    } else {
        Affine<F> v = load_affine<G>(a.aff, a.inf, a.n, hi);
        t = v.inf ? Jac<F>::identity() : Jac<F>{v.x, v.y, F::one()};
    }
    store_jac_soa<G>(a.jac, a.n, lo, jac_madd(t, u));
    t.Y = fp_neg(t.Y);
    store_jac_soa<G>(a.jac, a.n, hi, jac_madd(t, u));
}

// h_i = P_(i+m) - P_i for i < count (= m - 1); `aff` holds at least m + count decoded points
template <class G>
__global__ void __launch_bounds__(128) k_h_query(const uint32_t* aff, const uint8_t* inf, uint64_t m, uint64_t count,
                                                 uint32_t* jac) {
    using F = typename G::F;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    Affine<F> hi = load_affine<G>(aff, inf, 0, i + m);
    Affine<F> lo = affine_neg(load_affine<G>(aff, inf, 0, i));
    Jac<F> t = hi.inf ? Jac<F>::identity() : Jac<F>{hi.x, hi.y, F::one()};
    store_jac_soa<G>(jac, count, i, jac_madd(t, lo));
}

struct FftOps {
    void (*prepare)(int log_n, uint32_t* seq, uint32_t* ninv_m, cudaStream_t);
    void (*bitrev)(const uint32_t* src, const uint8_t* src_inf, uint32_t* dst, uint8_t* dst_inf, int log_n, cudaStream_t);
    void (*butterfly)(const ButterflyArgs&, cudaStream_t);
    void (*h_query)(const uint32_t* aff, const uint8_t* inf, uint64_t m, uint64_t count, uint32_t* jac, cudaStream_t);
    int max_log_n;  // two-adicity of the scalar field
};

template <class G>
struct FftLaunch {
    using FrP = typename G::Fr::Params;
    static void prepare(int log_n, uint32_t* seq, uint32_t* ninv_m, cudaStream_t s) {
        k_fft_prepare<FrP><<<1, 32, 0, s>>>(log_n, seq, ninv_m);
    }
    static void bitrev(const uint32_t* src, const uint8_t* src_inf, uint32_t* dst, uint8_t* dst_inf, int log_n,
                       cudaStream_t s) {
        constexpr int V = 2 * FieldWords<typename G::F>::W / 4;
        const uint64_t t = ((uint64_t)1 << log_n) * V;
        k_fft_bitrev<G><<<(unsigned)((t + 255) / 256), 256, 0, s>>>(src, src_inf, dst, dst_inf, log_n);
    }
    static void butterfly(const ButterflyArgs& a, cudaStream_t s) {
        const uint64_t half = a.n >> 1;
        if (!half) return;
        k_fft_butterfly<G><<<(unsigned)((half + 127) / 128), 128, 0, s>>>(a);
    }
    static void h_query(const uint32_t* aff, const uint8_t* inf, uint64_t m, uint64_t count, uint32_t* jac,
                        cudaStream_t s) {
        if (!count) return;
        k_h_query<G><<<(unsigned)((count + 127) / 128), 128, 0, s>>>(aff, inf, m, count, jac);
    }
    static FftOps ops() { return FftOps{&prepare, &bitrev, &butterfly, &h_query, FrP::TWO_ADICITY}; }
};

const FftOps& fft_ops_bls377_g1();
const FftOps& fft_ops_bls377_g2();
const FftOps& fft_ops_bw6_g1();
const FftOps& fft_ops_bw6_g2();
const FftOps& fft_ops_mnt4_g1();
const FftOps& fft_ops_mnt4_g2();
const FftOps& fft_ops_mnt6_g1();
const FftOps& fft_ops_mnt6_g2();

}  // namespace ss
