// Kernel instantiations for Mnt6G2 (MNT4/6-753 are exposed by the reference, setup-utils/src/converters.rs:18-45): the
// generic kernels over a 24-limb field with a != 0 formulas and byte-granular serialisation.  Functional coverage, not
// a tuned path: no endomorphism, no pairing instantiations.  The bucket-MSM kernels of this group live in
// kern_mnt6_g2_msm.cu and its group-FFT / QAP kernels in kern_mnt6_g2_fft.cu (translation units compile in parallel).
#include "kernels.cuh"

namespace ss {
const GroupOps& ops_mnt6_g2() {
    static const GroupOps o = GroupLaunch<Mnt6G2>::ops();
    return o;
}
}  // namespace ss
