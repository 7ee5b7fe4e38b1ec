// mesh_sort.h — internal: sort a triangle soup, or bare keys, by 64-bit order keys (meshpost.cu, cub::DeviceRadixSort).
#pragma once
#include <cuda_runtime.h>
#include <cstddef>

// d_keys (ntri, destroyed), d_v (9 floats per triangle), d_c (9 bytes per triangle or null) -> d_v_out / d_c_out in ascending key
// order.  key_bits = number of significant low bits of the keys.  Returns 0 or a cudaError_t.
int b2_sort_triangles (cudaStream_t s, size_t ntri, int key_bits, unsigned long long* d_keys, const float* d_v, const unsigned char* d_c,
                       float* d_v_out, unsigned char* d_c_out);
// d_keys (n) -> d_keys_out in ascending order (key_bits low bits significant).  Returns 0 or a cudaError_t.
int b2_sort_keys (cudaStream_t s, size_t n, int key_bits, const unsigned long long* d_keys, unsigned long long* d_keys_out);
