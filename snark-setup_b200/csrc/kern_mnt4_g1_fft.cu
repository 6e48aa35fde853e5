// Group-FFT and QAP kernel instantiations for Mnt4G1 (coordinates over Fq): k_fft_butterfly, k_h_query and the
// QAP sums of fft.cuh / qap.cuh.  The twiddle and coefficient multiplications run on k_scalar_mul of kern_mnt4_g1.cu
// (double-and-add, no endomorphism).  The exceptional P = Q case of the additions doubles through jac_dbl_cold, which
// takes the a != 0 formula (CurveCoeffA in ec.cuh).  A translation unit of its own keeps nvcc compile times parallel.
#include "qap.cuh"

namespace ss {
const FftOps& fft_ops_mnt4_g1() {
    static const FftOps o = FftLaunch<Mnt4G1>::ops();
    return o;
}
const QapOps& qap_ops_mnt4_g1() {
    static const QapOps o = QapLaunch<Mnt4G1>::ops();
    return o;
}
}  // namespace ss
