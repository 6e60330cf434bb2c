// Warp-level TF32 tensor-core helpers shared by the graph-stack kernels (gcn_block.cu, gcn_stack*.cu, gcn_tile.cu).
//
// fp32 parity (<= 1e-4 abs vs the reference) is kept by the 3xTF32 operand split: x = hi + lo with hi
// exactly representable in TF32, and  a*b ~= lo_a*hi_b + hi_a*lo_b + hi_a*hi_b  (fp32 accumulate).
#pragma once
#include "common.cuh"

namespace gcgcn {

__device__ __forceinline__ float4 ld4g(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float2 ld2g(const float* p) { return *reinterpret_cast<const float2*>(p); }

__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
    hi = __float_as_uint(x) & 0xffffe000u;
    lo = __float_as_uint(x - __uint_as_float(hi));
}

__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// One warp: C[16 x 8*NT] += A[16 x 8*ksteps] * B[8*ksteps x 8*NT] with fp32-accurate 3xTF32.
//   A(m,k) = pa[m*lda + k]                       (m in [0,16))
//   B(k,n) = pb[k*ldb + n]  (BT = false)  or  pb[n*ldb + k]  (BT = true)          (n in [0, 8*NT))
// Fragment layout (PTX m16n8k8): g = lane/4, t = lane%4
//   a0=(g,t) a1=(g+8,t) a2=(g,t+4) a3=(g+8,t+4);  b0=(t,g) b1=(t+4,g);  c0=(g,2t) c1=(g,2t+1) c2=(g+8,2t) c3=(g+8,2t+1)
// All per-lane addresses are formed once; the K loop only bumps two pointers.
template <int NT, bool BT>
__device__ __forceinline__ void warp_gemm(float (&c)[NT][4], int ksteps, const float* __restrict__ pa, int lda,
                                          const float* __restrict__ pb, int ldb) {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const float* a_lo = pa + g * lda + t;            // row g
    const float* a_hi = a_lo + 8 * lda;              // row g + 8
    const float* b0 = BT ? pb + g * ldb + t : pb + t * ldb + g;
    const int b_k4 = BT ? 4 : 4 * ldb;               // k -> k + 4
    const int b_n8 = BT ? 8 * ldb : 8;               // next 8-column tile
    const int b_step = BT ? 8 : 8 * ldb;             // next K step
#pragma unroll 2
    for (int ks = 0; ks < ksteps; ++ks) {
        uint32_t ah[4], al[4];
        split_tf32(a_lo[0], ah[0], al[0]);
        split_tf32(a_hi[0], ah[1], al[1]);
        split_tf32(a_lo[4], ah[2], al[2]);
        split_tf32(a_hi[4], ah[3], al[3]);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            uint32_t bh[2], bl[2];
            split_tf32(b0[nt * b_n8], bh[0], bl[0]);
            split_tf32(b0[nt * b_n8 + b_k4], bh[1], bl[1]);
            mma_tf32(c[nt], al, bh);
            mma_tf32(c[nt], ah, bl);
            mma_tf32(c[nt], ah, bh);
        }
        a_lo += 8;
        a_hi += 8;
        b0 += b_step;
    }
}

template <int NT>
__device__ __forceinline__ void zero_frag(float (&c)[NT][4]) {
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int q = 0; q < 4; ++q) c[nt][q] = 0.f;
}

}  // namespace gcgcn
