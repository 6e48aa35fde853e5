// Sparse matrix x point-vector products of the phase-2 QAP evaluation (phase2/src/polynomial.rs:11-94;
// SURVEY.md §8f rank 4):   out_v = sum_{e in row v} coeff_e * bases[index_e]     (dot_product, :80-94)
//
// The reference multiplies every entry by its coefficient (`coeffs[ind].mul(coeff)`, full double-and-add) on
// rayon threads.  R1CS matrices are almost entirely +-1, so here the host splits the entries of a row block
// into unit entries (a mixed addition of +-bases[index] straight from the decoded affine scratch) and general
// entries (one gathered k_scalar_mul pass over the compacted list, GLV/GLS), and the sums are formed in two
// passes so that a row with millions of entries (the constant-one variable) does not serialise on one thread:
//   k_qap_segment_sum : one thread per segment (<= 256 entries of one row)      -> Jacobian partial sums
//   k_qap_row_sum     : one thread per group of <= 256 partial sums of a row    -> second-level partial sums
//   k_qap_row_sum     : one thread per row over its second-level sums           -> Jacobian row sums
// followed by the usual batch normalisation + serialisation (k_normalize_encode).
#pragma once
#include "fft.cuh"

namespace ss {

struct QapSegArgs {
    const uint32_t* aff;  // decoded bases
    const uint8_t* inf;
    const uint32_t* index;      // per entry: base index (unit entries) or position in `general` (general entries)
    const uint8_t* kind;        // per entry: 0 = +1, 1 = -1, 2 = general, 3 = zero coefficient
    const uint64_t* seg_start;  // [nseg + 1] entry offsets of the segments
    uint64_t nseg;
    const uint32_t* general;  // Jacobian SoA [3*FW][ngeneral] of coeff_e * bases[index_e]
    uint64_t ngeneral;
    uint32_t* partial;  // out: Jacobian SoA [3*FW][nseg]
};

template <class G>
__global__ void __launch_bounds__(128) k_qap_segment_sum(QapSegArgs a) {
    using F = typename G::F;
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.nseg) return;
    Jac<F> acc = Jac<F>::identity();
    for (uint64_t e = a.seg_start[s]; e < a.seg_start[s + 1]; e++) {
        const uint8_t kd = a.kind[e];
        if (kd < 2) {
            Affine<F> p = load_affine<G>(a.aff, a.inf, 0, a.index[e]);
            if (kd) p.y = fp_neg(p.y);
            acc = jac_madd(acc, p);
        } else if (kd == 2) {
            acc = jac_add(acc, load_jac_soa<G>(a.general, a.ngeneral, a.index[e]));
        }
    }
    store_jac_soa<G>(a.partial, a.nseg, s, acc);
}

// rows[v] = sum of partial[row_seg[v] .. row_seg[v+1])
template <class G>
__global__ void __launch_bounds__(128) k_qap_row_sum(const uint32_t* partial, uint64_t nseg, const uint64_t* row_seg,
                                                     uint64_t rows, uint32_t* out) {
    using F = typename G::F;
    const uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= rows) return;
    Jac<F> acc = Jac<F>::identity();
    for (uint64_t s = row_seg[v]; s < row_seg[v + 1]; s++) acc = jac_add(acc, load_jac_soa<G>(partial, nseg, s));
    store_jac_soa<G>(out, rows, v, acc);
}

struct QapOps {
    void (*segment_sum)(const QapSegArgs&, cudaStream_t);
    void (*row_sum)(const uint32_t* partial, uint64_t nseg, const uint64_t* row_seg, uint64_t rows, uint32_t* out, cudaStream_t);
};
template <class G>
struct QapLaunch {
    static void segment_sum(const QapSegArgs& a, cudaStream_t s) {
        if (a.nseg) k_qap_segment_sum<G><<<(unsigned)((a.nseg + 127) / 128), 128, 0, s>>>(a);
    }
    static void row_sum(const uint32_t* partial, uint64_t nseg, const uint64_t* row_seg, uint64_t rows, uint32_t* out,
                        cudaStream_t s) {
        if (rows) k_qap_row_sum<G><<<(unsigned)((rows + 127) / 128), 128, 0, s>>>(partial, nseg, row_seg, rows, out);
    }
    static QapOps ops() { return QapOps{&segment_sum, &row_sum}; }
};

const QapOps& qap_ops_bls377_g1();
const QapOps& qap_ops_bls377_g2();
const QapOps& qap_ops_bw6_g1();
const QapOps& qap_ops_bw6_g2();
const QapOps& qap_ops_mnt4_g1();
const QapOps& qap_ops_mnt4_g2();
const QapOps& qap_ops_mnt6_g1();
const QapOps& qap_ops_mnt6_g2();

}  // namespace ss
