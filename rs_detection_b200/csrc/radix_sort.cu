// radix_sort.cu -- the stable key/value radix sort of the deterministic RoIAlignRotated backward (roi_align.cu).
//
// A unit of its own so that CUB's kernels and device globals stay out of roi_align.cu's module.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace rsdet {

// Stable LSD radix sort of n (uint32 key, int32 value) pairs on bits [0, key_bits) of the key, ping-ponging between
// the A and B buffers.  tmp == nullptr: *tmp_bytes receives the temporary storage the sort needs, nothing is launched.
// Otherwise the sort is enqueued on `st` and *in_b tells whether the sorted pairs ended in the B buffers.
int sort_pairs_u32(void* tmp, size_t* tmp_bytes, uint32_t* key_a, uint32_t* key_b, int* val_a, int* val_b, int n, int key_bits,
                   bool* in_b, cudaStream_t st) {
    cub::DoubleBuffer<uint32_t> dk(key_a, key_b);
    cub::DoubleBuffer<int> dv(val_a, val_b);
    const cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp, *tmp_bytes, dk, dv, n, 0, key_bits, st);
    if (in_b) *in_b = dk.Current() == key_b;
    return e == cudaSuccess ? RSDET_OK : (int)e;
}

}  // namespace rsdet
