// rtb_tail.cu — the 32 instantiations of tail_kernel of one (MEDIA, stack), one per feature word (rtb_kernels.h).  The
// Makefile compiles this file once per (TAIL_MEDIA, TAIL_DEEP) into objects of their own, so that they compile in parallel.
#include <utility>

#include "rtb_device.h"

namespace rtb {

template <bool MEDIA, int STACK, uint32_t... F>
static TailKernel tail_kernel_of(uint32_t f, std::integer_sequence<uint32_t, F...>) {
	static const TailKernel table[] = {tail_kernel<MEDIA, STACK, F>...};
	return table[f];
}

template <bool MEDIA, bool DEEP>
TailKernel tail_kernel_for(uint32_t f) {
	return tail_kernel_of<MEDIA, DEEP ? DEEP_STACK_SIZE : STACK_SIZE>(f, std::make_integer_sequence<uint32_t, F_WORDS>());
}
template TailKernel tail_kernel_for<TAIL_MEDIA, TAIL_DEEP>(uint32_t f);

}  // namespace rtb
