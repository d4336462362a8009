// Test tool: the signature subgroup test of blsgpu_verify_batch's split path on single points, built with g++ (-x c++) for the host and
// with nvcc for sm_100a from this one source.  Per point q (affine Montgomery limbs x.c0, x.c1, y.c0, y.c1): the doubling / addition
// steps pair (-g1, q) runs in k_miller_lines over all of its launches, then out[0] = miller_end_in_subgroup on the end point,
// out[1] = the end point's Z is 0, out[2] = g2_in_subgroup(q), the decoder's test.
#include "stages.cuh"
using namespace bls;

BLS_HD void end_point_check(const fp* in, uint32_t* out) {
    g2_aff q; q.x.c0 = in[0]; q.x.c1 = in[1]; q.y.c0 = in[2]; q.y.c1 = in[3];
    g2_proj r; r.x = q.x; r.y = q.y; r.z = fp2_one();
    const uint64_t x = BLS_X_ABS; fp2 c0, c1, c2;
    for (int it = 62; it >= 0; it--) {
        miller_dbl(r, c0, c1, c2);
        if ((x >> it) & 1) miller_add(r, q, c0, c1, c2);
    }
    out[0] = miller_end_in_subgroup(r, q) ? 1u : 0u; out[1] = fp2_is_zero(r.z) ? 1u : 0u; out[2] = g2_in_subgroup(q) ? 1u : 0u;
}

#if defined(__CUDACC__)
__global__ void __launch_bounds__(128, 2) k_end_point_check(const fp* in, size_t n, uint32_t* out) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    end_point_check(in + 4 * i, out + 3 * i);
}
extern "C" int dev_end_point_check(const uint8_t* in, size_t n, uint32_t* out) {
    fp* din; uint32_t* dout;
    if (cudaMalloc(&din, 192 * n) != cudaSuccess) return -2;
    if (cudaMalloc(&dout, 12 * n) != cudaSuccess) { cudaFree(din); return -2; }
    cudaMemcpy(din, in, 192 * n, cudaMemcpyHostToDevice);
    k_end_point_check<<<(unsigned)((n + 127) / 128), 128>>>(din, n, dout);
    cudaError_t e = cudaDeviceSynchronize();
    cudaMemcpy(out, dout, 12 * n, cudaMemcpyDeviceToHost); cudaFree(din); cudaFree(dout);
    return e == cudaSuccess ? 0 : -3;
}
#else
extern "C" int host_end_point_check(const uint8_t* in, size_t n, uint32_t* out) {
    for (size_t i = 0; i < n; i++) end_point_check(reinterpret_cast<const fp*>(in) + 4 * i, out + 3 * i);
    return 0;
}
#endif
