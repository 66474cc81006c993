// rtb_shade.cu — the 32 instantiations of shade_kernel, one per feature word (rtb_kernels.h), in an object of their own
// so that they compile in parallel with the other kernel objects.
#include <utility>

#include "rtb_device.h"

namespace rtb {

template <uint32_t... F>
static ShadeKernel shade_kernel_of(uint32_t f, std::integer_sequence<uint32_t, F...>) {
	static const ShadeKernel table[] = {shade_kernel<F>...};
	return table[f];
}

ShadeKernel shade_kernel_for(uint32_t f) { return shade_kernel_of(f, std::make_integer_sequence<uint32_t, F_WORDS>()); }

}  // namespace rtb
