// tools/pcie_probe_multi.cu — what the host links of this box do when 1, 2, 4, 8 GPUs copy AT THE SAME TIME: the
// ceiling the end-to-end (host arrays in / host arrays out) leg of bench.py runs against at N > 1.
//   mkdir -p build && nvcc -O2 -std=c++17 -o build/pcie_probe_multi tools/pcie_probe_multi.cu -lpthread
//   build/pcie_probe_multi [--gb 1.0] [--wc] [--bind] [--max-gpus 8]
// One host thread per GPU; every thread allocates its own pinned buffers AFTER cudaSetDevice (and, with --bind, after
// pinning itself to the CPUs of the GPU's NUMA node, so first touch places the pages there); --wc allocates the
// host->device source write-combined. Each configuration is timed between two barriers (wall clock, max over
// threads), best of 3. Prints one JSON line per (gpus, direction) with per-GPU and aggregate GB/s.
#include <cuda_runtime.h>
#include <pthread.h>
#include <sched.h>

#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <string>
#include <thread>
#include <vector>

static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct Barrier {
  pthread_barrier_t b;
  explicit Barrier(int n) { pthread_barrier_init(&b, nullptr, n); }
  void wait() { pthread_barrier_wait(&b); }
};

// CPUs of the NUMA node the GPU hangs off (sysfs), or empty
static std::vector<int> cpus_of_gpu(int dev) {
  std::vector<int> out;
  char bdf[32] = "";
  if (cudaDeviceGetPCIBusId(bdf, sizeof bdf, dev) != cudaSuccess) return out;
  for (char* p = bdf; *p; ++p) *p = (char)tolower(*p);
  std::ifstream f(std::string("/sys/bus/pci/devices/") + bdf + "/numa_node");
  int node = -1;
  if (!(f >> node) || node < 0) return out;
  std::ifstream c("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
  std::string list;
  if (!(c >> list)) return out;
  size_t pos = 0;
  while (pos < list.size()) {
    size_t end = list.find(',', pos);
    if (end == std::string::npos) end = list.size();
    const std::string part = list.substr(pos, end - pos);
    const size_t dash = part.find('-');
    const int a = atoi(part.c_str()), b = dash == std::string::npos ? a : atoi(part.c_str() + dash + 1);
    for (int i = a; i <= b; ++i) out.push_back(i);
    pos = end + 1;
  }
  return out;
}

int main(int argc, char** argv) {
  double gb = 1.0;
  bool wc = false, bind = false;
  int max_gpus = 8;
  for (int i = 1; i < argc; ++i) {
    if (!strcmp(argv[i], "--gb") && i + 1 < argc) gb = atof(argv[++i]);
    else if (!strcmp(argv[i], "--wc")) wc = true;
    else if (!strcmp(argv[i], "--bind")) bind = true;
    else if (!strcmp(argv[i], "--max-gpus") && i + 1 < argc) max_gpus = atoi(argv[++i]);
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
    printf("{\"error\": \"no CUDA device\"}\n");
    return 1;
  }
  if (ndev > max_gpus) ndev = max_gpus;
  const size_t bytes = (size_t)(gb * (1u << 30));
  printf("{\"probe\": \"pcie_probe_multi\", \"gpus_visible\": %d, \"bytes_per_copy\": %zu, \"write_combined\": %s, \"numa_bind\": %s, "
         "\"host_threads\": %u}\n", ndev, bytes, wc ? "true" : "false", bind ? "true" : "false", std::thread::hardware_concurrency());
  for (int G = 1; G <= ndev; G *= 2) {
    for (int mode = 0; mode < 3; ++mode) {  // 0 h2d, 1 d2h, 2 both
      Barrier bar(G + 1);
      std::vector<double> t_thread(G, 0.0);
      std::atomic<int> failed{0};
      std::vector<int> nodes_cpus(G, 0);
      std::vector<std::thread> th;
      double best = 1e30;
      for (int g = 0; g < G; ++g)
        th.emplace_back([&, g] {
          if (bind) {
            const std::vector<int> cpus = cpus_of_gpu(g);
            if (!cpus.empty()) {
              cpu_set_t set;
              CPU_ZERO(&set);
              for (int c : cpus) CPU_SET(c, &set);
              sched_setaffinity(0, sizeof set, &set);
              nodes_cpus[g] = (int)cpus.size();
            }
          }
          char *h_in = nullptr, *h_out = nullptr, *d_in = nullptr, *d_out = nullptr;
          cudaStream_t s1, s2;
          bool ok = cudaSetDevice(g) == cudaSuccess;
          ok = ok && cudaHostAlloc(&h_in, bytes, wc ? cudaHostAllocWriteCombined : cudaHostAllocDefault) == cudaSuccess;
          ok = ok && cudaHostAlloc(&h_out, bytes, cudaHostAllocDefault) == cudaSuccess;
          ok = ok && cudaMalloc(&d_in, bytes) == cudaSuccess && cudaMalloc(&d_out, bytes) == cudaSuccess;
          ok = ok && cudaStreamCreate(&s1) == cudaSuccess && cudaStreamCreate(&s2) == cudaSuccess;
          if (ok) {
            memset(h_in, 1, bytes);
            memset(h_out, 2, bytes);
          } else {
            failed = 1;
          }
          for (int rep = 0; rep < 4; ++rep) {  // rep 0 = warm-up
            if (ok) cudaDeviceSynchronize();
            bar.wait();
            const double t0 = now();
            if (ok) {
              if (mode != 1) cudaMemcpyAsync(d_in, h_in, bytes, cudaMemcpyHostToDevice, s1);
              if (mode != 0) cudaMemcpyAsync(h_out, d_out, bytes, cudaMemcpyDeviceToHost, s2);
              cudaDeviceSynchronize();
            }
            t_thread[g] = now() - t0;
            bar.wait();
            bar.wait();
          }
          if (h_in) cudaFreeHost(h_in);
          if (h_out) cudaFreeHost(h_out);
          if (d_in) cudaFree(d_in);
          if (d_out) cudaFree(d_out);
        });
      for (int rep = 0; rep < 4; ++rep) {
        bar.wait();
        bar.wait();
        double worst = 0;
        for (double t : t_thread) worst = t > worst ? t : worst;
        if (rep > 0 && worst < best) best = worst;
        bar.wait();
      }
      for (auto& t : th) t.join();
      const char* name = mode == 0 ? "h2d" : mode == 1 ? "d2h" : "duplex";
      const double per = bytes / best / 1e9;
      printf("{\"gpus\": %d, \"direction\": \"%s\", \"per_gpu_gbs_each_direction\": %.2f, \"aggregate_gbs_each_direction\": %.2f, "
             "\"failed\": %d, \"cpus_bound_gpu0\": %d}\n", G, name, per, per * G, failed.load(), nodes_cpus[0]);
      fflush(stdout);
    }
  }
  return 0;
}
