// csc_lab.cu — standalone timing and per-CTA trace of the library's CSC launch (tools only; not part of libb2video.so).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -DCSC_TRACE -o tools/lab/csc_lab tools/lab/csc_lab.cu
// Run on the GPU box: tools/lab/csc_lab [w h]
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

__device__ unsigned long long* g_trace;    // [cta][4]: start ns, end ns, smid, unused
#include "../../selkies_b200/csrc/csc.cu"

using namespace b2v;

static void summarize(const char* name, std::vector<unsigned long long>& tr, int ctas) {
  unsigned long long t0 = ~0ull, t1 = 0;
  for (int i = 0; i < ctas; i++) { t0 = std::min(t0, tr[4 * i]); t1 = std::max(t1, tr[4 * i + 1]); }
  std::vector<double> st, en;
  std::vector<double> sm_first(256, 1e18), sm_last(256, 0);
  for (int i = 0; i < ctas; i++) {
    st.push_back((tr[4 * i] - t0) * 1e-3); en.push_back((tr[4 * i + 1] - t0) * 1e-3);
    int sm = (int)tr[4 * i + 2];
    sm_first[sm] = std::min(sm_first[sm], st.back()); sm_last[sm] = std::max(sm_last[sm], en.back());
  }
  std::sort(st.begin(), st.end()); std::sort(en.begin(), en.end());
  double act = 0; int nsm = 0; double lastmin = 1e18, lastmax = 0;
  for (int s = 0; s < 256; s++) if (sm_last[s] > 0) { act += sm_last[s] - sm_first[s]; nsm++; lastmin = std::min(lastmin, sm_last[s]); lastmax = std::max(lastmax, sm_last[s]); }
  printf("%-22s ctas %5d span %.2f us | CTA start p0 %.2f p50 %.2f p90 %.2f p100 %.2f | CTA end p0 %.2f p10 %.2f p50 %.2f p100 %.2f | SMs %d mean busy span %.2f, SM finish min %.2f max %.2f\n",
         name, ctas, (t1 - t0) * 1e-3, st[0], st[ctas / 2], st[ctas * 9 / 10], st[ctas - 1], en[0], en[ctas / 10], en[ctas / 2], en[ctas - 1], nsm, act / nsm, lastmin, lastmax);
}

// leaves L2 full of DIRTY lines, like the encoder kernels that run between two CSC launches of the real pipeline
__global__ void k_pollute(uint4* buf, size_t n16) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) { uint4 v = buf[i]; v.x += 1; v.y ^= v.x; buf[i] = v; }
}

int main(int argc, char** argv) {
  int w = argc > 2 ? atoi(argv[1]) : 3840, h = argc > 2 ? atoi(argv[2]) : 2160;
  const int NF = 8;
  size_t fb = (size_t)w * h * 4, ob = (size_t)w * h * 3 / 2;
  std::vector<uint8_t*> in(NF), out(NF);
  std::vector<uint8_t> host(fb);
  for (size_t i = 0; i < fb; i++) host[i] = (uint8_t)(rand() >> 7);
  for (int i = 0; i < NF; i++) { cudaMalloc(&in[i], fb); cudaMalloc(&out[i], ob); cudaMemcpy(in[i], host.data(), fb, cudaMemcpyHostToDevice); }
  unsigned long long* d_tr; const int MAXC = 1 << 16;
  cudaMalloc(&d_tr, MAXC * 4 * 8);
  cudaMemcpyToSymbol(g_trace, &d_tr, sizeof d_tr);
  cudaStream_t st; cudaStreamCreate(&st);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  auto params = [&](int i) {
    CscParams p{}; p.src = in[i]; p.src_w = w; p.src_h = h; p.src_stride = w * 4; p.dst_w = w; p.dst_h = h; p.coded_w = w; p.coded_h = h;
    p.out_y = out[i]; p.out_uv = out[i] + (size_t)w * h; return p;
  };
  const char* name = "csc_bgra_nv12_fast";
  for (int i = 0; i < NF; i++) launch_csc(params(i), st);
  cudaStreamSynchronize(st);
  cudaEventRecord(e0, st);
  const int IT = 200;
  for (int i = 0; i < IT; i++) launch_csc(params(i % NF), st);
  cudaEventRecord(e1, st); cudaStreamSynchronize(st);
  float ms; cudaEventElapsedTime(&ms, e0, e1);
  double us = ms * 1e3 / IT;
  printf("%-22s %dx%d burst %.2f us/launch = %.0f GB/s algorithmic (%s)\n", name, w, h, us, w * h * 5.5 / us * 1e-3, cudaGetErrorString(cudaGetLastError()));
  // traced launches: (a) after an idle device, (b) after a kernel that left ~96 MB of dirty lines in L2, (c) same + 100 us of idle
  uint4* pol = nullptr; const size_t pol_bytes = 96u << 20;
  cudaMalloc(&pol, pol_bytes); cudaMemset(pol, 1, pol_bytes);
  for (int mode = 1; mode <= 2; mode++) {
    cudaMemset(d_tr, 0, MAXC * 4 * 8);
    cudaDeviceSynchronize();
    k_pollute<<<148 * 8, 256, 0, st>>>(pol, pol_bytes / 16);
    if (mode == 2) { cudaStreamSynchronize(st); }
    launch_csc(params(5), st);
    cudaStreamSynchronize(st);
    std::vector<unsigned long long> tr2(MAXC * 4);
    cudaMemcpy(tr2.data(), d_tr, MAXC * 4 * 8, cudaMemcpyDeviceToHost);
    int c2 = 0; while (c2 < MAXC && tr2[4 * c2]) c2++;
    char nm[64]; snprintf(nm, 64, "%s %s", name, mode == 1 ? "after-dirty-L2" : "dirty-L2+sync");
    if (c2) summarize(nm, tr2, c2);
  }
  cudaMemset(d_tr, 0, MAXC * 4 * 8);
  cudaDeviceSynchronize();
  launch_csc(params(3), st);
  cudaStreamSynchronize(st);
  std::vector<unsigned long long> tr(MAXC * 4);
  cudaMemcpy(tr.data(), d_tr, MAXC * 4 * 8, cudaMemcpyDeviceToHost);
  int ctas = 0; while (ctas < MAXC && tr[4 * ctas]) ctas++;
  if (ctas) summarize(name, tr, ctas);
  return 0;
}
