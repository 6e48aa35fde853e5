// Kernel instantiations for Mnt4G1 (MNT4/6-753 are exposed by the reference, setup-utils/src/converters.rs:18-45): the
// generic kernels over a 24-limb field with a != 0 formulas and byte-granular serialisation.  Functional coverage, not
// a tuned path: no endomorphism, no pairing instantiations; the group-FFT / QAP kernels are in kern_mnt4_g1_fft.cu.
#include "msm.cuh"

namespace ss {
const GroupOps& ops_mnt4_g1() {
    static const GroupOps o = GroupLaunch<Mnt4G1>::ops();
    return o;
}
const MsmOps& msm_ops_mnt4_g1() {
    static const MsmOps o = MsmLaunch<Mnt4G1>::ops();
    return o;
}
}  // namespace ss
