// tools/pcie_probe.cu — what the host link of this box can do: 1-D and pitched (one time level out of three)
// copies, each direction alone and both at once. Development probe for caar_run_host's pipeline.
//   mkdir -p build && nvcc -O2 -o build/pcie_probe tools/pcie_probe.cu && build/pcie_probe
#include <cuda_runtime.h>
#include <chrono>
#include <cstdio>
#include <cstring>
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); return 1; } } while (0)
static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
int main() {
  const size_t rows = 40000, width = 9216 * 2, pitch = width * 3;  // v: 18432 B of every 55296 B
  const size_t bytes = rows * pitch;                                // 2.2 GB
  char *h_in, *h_out, *d_in, *d_out;
  CK(cudaMallocHost(&h_in, bytes)); CK(cudaMallocHost(&h_out, bytes));
  CK(cudaMalloc(&d_in, bytes)); CK(cudaMalloc(&d_out, bytes));
  memset(h_in, 1, bytes); memset(h_out, 2, bytes);
  cudaStream_t s1, s2; CK(cudaStreamCreate(&s1)); CK(cudaStreamCreate(&s2));
  size_t rows_v = rows, width_v = width, pitch_v = pitch;
  auto run = [&](const char* name, int in_mode, int out_mode) {  // 0 none, 1 = 1-D (same byte count), 2 = pitched
    const size_t rows = rows_v, width = width_v, pitch = pitch_v;
    const size_t moved = rows * width;
    double best = 1e9;
    for (int rep = 0; rep < 3; ++rep) {
      cudaDeviceSynchronize();
      const double t0 = now();
      for (int part = 0; part < 8; ++part) {  // 8 chunks like the pipeline
        const size_t r0 = rows / 8 * part, nr = rows / 8;
        if (in_mode == 1) cudaMemcpyAsync(d_in + r0 * width, h_in + r0 * width, nr * width, cudaMemcpyHostToDevice, s1);
        if (in_mode == 2) cudaMemcpy2DAsync(d_in + r0 * pitch, pitch, h_in + r0 * pitch, pitch, width, nr, cudaMemcpyHostToDevice, s1);
        if (out_mode == 1) cudaMemcpyAsync(h_out + r0 * width, d_out + r0 * width, nr * width, cudaMemcpyDeviceToHost, s2);
        if (out_mode == 2) cudaMemcpy2DAsync(h_out + r0 * pitch, pitch, d_out + r0 * pitch, pitch, width, nr, cudaMemcpyDeviceToHost, s2);
      }
      cudaDeviceSynchronize();
      const double dt = now() - t0;
      if (dt < best) best = dt;
    }
    printf("%-34s h2d %6.2f GB/s   d2h %6.2f GB/s\n", name, in_mode ? moved / best / 1e9 : 0.0, out_mode ? moved / best / 1e9 : 0.0);
    return 0;
  };
  run("h2d 1-D alone", 1, 0);
  run("h2d pitched alone", 2, 0);
  run("d2h 1-D alone", 0, 1);
  run("d2h pitched alone", 0, 2);
  run("both 1-D", 1, 1);
  run("both pitched", 2, 2);
  run("h2d pitched + d2h 1-D", 2, 1);
  run("h2d 1-D + d2h pitched", 1, 2);
  // one level-field rows (9216 B of 27648 B), as dp3d / T
  rows_v = 80000; width_v = 9216; pitch_v = 27648;
  run("both pitched, 9 KB rows", 2, 2);
  // long rows: 1.1 MB of every 3.3 MB
  rows_v = 664; width_v = 18432 * 60; pitch_v = width_v * 3;
  run("both pitched, 1.1 MB rows", 2, 2);
  rows_v = 8 * 1296; width_v = 18432 * 4; pitch_v = width_v * 3;
  run("both pitched, 72 KB rows", 2, 2);
  return 0;
}
