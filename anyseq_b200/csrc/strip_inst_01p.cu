// packed-cell strip kernels: global / semiglobal Gotoh, column masks, two-row tiles (strip_packed.cuh)
#include "strip_kernel.cuh"

namespace anyseq {

StripKernelFn get_strip_kernel_01p(int K)
{
    switch (K) {
        case 16: return strip_kernel<false, true, 16, true, false, 3>;
        case 32: return strip_kernel<false, true, 32, true, false, 3>;
        default: return nullptr;
    }
}

}  // namespace anyseq
