// Device unit-test library (TEST TOOL ONLY): applies one primitive of the CUDA device library per thread.
#include <cuda_runtime.h>
#include <cstdlib>
#include "ops.h"
#include "coop.cuh"
using namespace bls;
// one kernel per primitive (template instantiation): keeps each kernel small -- a single kernel holding all cases behind a
// run-time switch (10 KB frame, ~1 MB of code) was itself miscompiled by nvcc 12.9 (inputs of some cases read back as garbage).
template <int OP> __global__ void __launch_bounds__(128, 2) k_run_op(const fp* in, fp* out, size_t n, int n_in, int n_out) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    fp a[24], r[24];
    for (int k = 0; k < n_in; k++) a[k] = in[i * n_in + k];
    for (int k = 0; k < n_out; k++) r[k] = fp_zero();
    run_op(OP, a, r);
    for (int k = 0; k < n_out; k++) out[i * n_out + k] = r[k];
}
template <int OP> static void launch(const fp* din, fp* dout, size_t n, op_desc d) { k_run_op<OP><<<(unsigned)((n + 127) / 128), 128>>>(din, dout, n, d.n_in, d.n_out); }
extern "C" int dev_run_op(int op, const uint8_t* in, uint8_t* out, size_t n) {
    op_desc d = op_shape(op); if (!d.n_in) return -1;
    fp *din, *dout; size_t bi = n * d.n_in * 48, bo = n * d.n_out * 48;
    if (cudaMalloc(&din, bi) != cudaSuccess || cudaMalloc(&dout, bo) != cudaSuccess) return -2;
    cudaMemcpy(din, in, bi, cudaMemcpyHostToDevice);
    switch (op) {
#define L(K) case K: launch<K>(din, dout, n, d); break;
        L(1) L(2) L(3) L(4) L(5) L(6) L(7) L(8) L(9) L(10) L(11) L(12) L(13) L(14) L(15) L(16) L(17) L(18) L(19) L(20) L(21) L(22) L(23) L(24) L(25) L(26) L(27) L(28) L(29) L(30) L(31) L(32) L(33) L(34) L(35) L(36) L(37) L(38) L(39) L(40) L(41) L(42) L(43) L(44) L(45) L(46)
#undef L
        default: cudaFree(din); cudaFree(dout); return -1;
    }
    cudaError_t e = cudaDeviceSynchronize();
    cudaMemcpy(out, dout, bo, cudaMemcpyDeviceToHost); cudaFree(din); cudaFree(dout);
    return e == cudaSuccess ? 0 : -3;
}

// ---- throughput ladder (profiles/r01_tuning.md): `reps` dependent applications of one primitive per thread, output fed back
template <int OP> __global__ void __launch_bounds__(128, 2) k_bench_op(const fp* in, fp* out, size_t n, int n_in, int n_out, int reps) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    fp a[24], r[24];
    for (int k = 0; k < n_in; k++) a[k] = in[i * n_in + k];
    for (int k = 0; k < n_out; k++) r[k] = fp_zero();
    for (int it = 0; it < reps; it++) { run_op(OP, a, r); for (int k = 0; k < n_out && k < n_in; k++) a[k] = r[k]; }
    for (int k = 0; k < n_out; k++) out[i * n_out + k] = r[k];
}
template <int OP> static void launch_bench(const fp* din, fp* dout, size_t n, op_desc d, int reps) { k_bench_op<OP><<<(unsigned)((n + 127) / 128), 128>>>(din, dout, n, d.n_in, d.n_out, reps); }
extern "C" float dev_bench_op(int op, size_t n, int reps) {
    op_desc d = op_shape(op); if (!d.n_in) return -1.f;
    fp *din, *dout; size_t bi = n * d.n_in * 48, bo = n * d.n_out * 48;
    if (cudaMalloc(&din, bi) != cudaSuccess || cudaMalloc(&dout, bo) != cudaSuccess) return -2.f;
    cudaMemset(din, 0x11, bi);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1); float best = 1e30f;
    for (int r = 0; r < 3; r++) {
        cudaEventRecord(e0);
        switch (op) {
#define L(K) case K: launch_bench<K>(din, dout, n, d, reps); break;
            L(21) L(1) L(2) L(3) L(8) L(9) L(10) L(11) L(12) L(5) L(6) L(29) L(30) L(31) L(32) L(33) L(34) L(35)
#undef L
            default: return -1.f;
        }
        cudaEventRecord(e1); cudaEventSynchronize(e1); float ms; cudaEventElapsedTime(&ms, e0, e1); if (r && ms < best) best = ms;
    }
    cudaFree(din); cudaFree(dout);
    return best;
}


// cooperative Fp12 primitives: dependent chain of coop_mul / coop_cyclo_sqr, 5 items per warp
__global__ void __launch_bounds__(128, 2) k_coop_bench(fp* out, int reps, int which) {
    __shared__ coop_smem sm[4];
    coop_lane c = coop_init(&sm[threadIdx.x >> 5]);
    fp2 r, b; r.c0 = fp_one(); r.c1 = fp_zero(); r.c0.l[0] ^= threadIdx.x; b = r; b.c1.l[1] = 77u + c.k;
    for (int it = 0; it < reps; it++) r = which == 0 ? coop_mul(c, r, b) : coop_cyclo_sqr(c, r);
    if (r.c0.l[0] == 0x12345u) out[0] = r.c0;
}
extern "C" float dev_coop_bench(int which, int warps_per_smsp, int reps) {
    fp* dout; cudaMalloc(&dout, 4096);
    int sms = 0; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1); float best = 1e30f;
    for (int r = 0; r < 3; r++) {
        cudaEventRecord(e0); k_coop_bench<<<sms * warps_per_smsp, 128>>>(dout, reps, which); cudaEventRecord(e1); cudaEventSynchronize(e1);
        float ms; cudaEventElapsedTime(&ms, e0, e1); if (r && ms < best) best = ms;
    }
    cudaFree(dout); return best;
}

extern "C" void dev_op_shape(int op, int* n_in, int* n_out) { op_desc d = op_shape(op); *n_in = d.n_in; *n_out = d.n_out; }
