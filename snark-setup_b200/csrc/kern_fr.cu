// Scalar-field inversion on the device (phase 2's delta^-1, MPCParameters::contribute, phase2/src/parameters.rs:294-296).
// A translation unit of its own, so that the group kernels' objects are not touched by it.
#include "kernels.cuh"

namespace ss {

// out = a^-1, both Montgomery (the fp_inv of k_marlin_scalars); one thread
template <class FrP>
__global__ void k_fr_inverse(const uint32_t* a, uint32_t* out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    Fp<FrP> x;
    for (int i = 0; i < FrP::N; i++) x.l[i] = a[i];
    const Fp<FrP> y = fp_inv(x);
    for (int i = 0; i < FrP::N; i++) out[i] = y.l[i];
}

// curve ids of include/snark_setup_b200.h (ss_curve)
void fr_inverse(int curve, const uint32_t* a_mont, uint32_t* out_mont, cudaStream_t s) {
    switch (curve) {
        case 0: k_fr_inverse<Bls377Fr><<<1, 32, 0, s>>>(a_mont, out_mont); break;
        case 1: k_fr_inverse<Bls377Fq><<<1, 32, 0, s>>>(a_mont, out_mont); break;  // BW6-761 Fr = BLS12-377 Fq
        case 2: k_fr_inverse<Mnt753R><<<1, 32, 0, s>>>(a_mont, out_mont); break;
        case 3: k_fr_inverse<Mnt753Q><<<1, 32, 0, s>>>(a_mont, out_mont); break;
    }
}

}  // namespace ss
