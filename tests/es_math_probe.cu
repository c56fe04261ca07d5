// TEST INFRASTRUCTURE -- applies the library's device es_log (op 0) or es_exp (op 1) to n doubles, so that tests can
// compare them with the oracle's sbo_det_log / sbo_det_exp bit for bit.  tests/test_exact_math.py compiles it at run
// time with the library's NVCC_FLAGS.
#include "sb_es.cuh"

__global__ void k_es_math_probe(int n, int op, const double* x, double* y) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = op == 0 ? es_log(x[i]) : es_exp(x[i]);
}

// x_host, y_host: n doubles on the host.  Returns 0 or the first CUDA error.
extern "C" int es_math_probe(int n, int op, const double* x_host, double* y_host) {
  double *x = nullptr, *y = nullptr;
  const size_t bytes = sizeof(double) * (size_t)n;
  cudaError_t e = cudaMalloc(&x, bytes);
  if (e == cudaSuccess) e = cudaMalloc(&y, bytes);
  if (e == cudaSuccess) e = cudaMemcpy(x, x_host, bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    k_es_math_probe<<<(n + 127) / 128, 128>>>(n, op, x, y);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpy(y_host, y, bytes, cudaMemcpyDeviceToHost);
  cudaFree(x);
  cudaFree(y);
  return (int)e;
}
