/* swinb200_debug -- bring-up hooks of libswinb200.so.  NOT part of the drop-in boundary (include/swinb200.h): nothing in
 * the package's hot path calls these; tools/ and a few kernel tests do. */
#ifndef SWINB200_DEBUG_H_
#define SWINB200_DEBUG_H_

#ifdef __cplusplus
extern "C" {
#endif

/* D[128,N] (fp32) = A[128,K] * B[N,K]^T through one tcgen05.mma chain using the un-swizzled core-matrix
 * shared-memory layout of the attention kernels.  a_mode: 0 = A (128,K) from smem K-major, 1 = A stored (K,128)
 * from smem M-major, 2 = A (128,K) from tensor memory;  b_mode: 0 = B stored (N,K), 1 = B stored (K,N).
 * pad16: extra 16-byte units added to the chunk stride.  No reference counterpart. */
int swinb200_debug_umma_probe(const void* A, const void* B, float* D, int N, int K, int a_mode, int b_mode,
                              int pad16, void* stream);

/* bring-up aid: when buf != NULL the tcgen05 attention backward at 9x18 windows / head_dim 96 writes the clock64() cycles
 * each CTA < 4096 spent per phase into buf[cta*16 + phase] (int64).  Pass NULL to switch it off. */
int swinb200_debug_attn_phase_buffer(void* buf);

#ifdef __cplusplus
}
#endif
#endif /* SWINB200_DEBUG_H_ */
