// fused inverse STFT kernels: FFT sizes 64..8192 (core M = 32..4096), on the core plans of the forward STFT variants
// (wfb_variants_f32_stft.cu): the span kernel's plan, pad quantum and frames per tile from N = 256, the direct kernel's
// plan with 128 threads per CTA below
#include "wfb_registry.h"
namespace wfb {
#define V(PL, X, PQ, MINB) IstftLaunchers<PL, X, PQ, MINB>::make(#PL "_istft" #X)
const std::vector<IstftVariant> &variants_istft() {
    static const std::vector<IstftVariant> v = {
        V(F32_32, 64, 16, 2), V(F32_64, 32, 16, 2),
        V(F32_128, 16, 16, 3), V(F32_256, 8, 16, 3), V(P32_512, 8, 16, 3),
        V(P32_1024, 4, 32, 3), V(F32_2048, 2, 16, 2), V(F32_4096, 2, 16, 1),
    };
    return v;
}
}  // namespace wfb
