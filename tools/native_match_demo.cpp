// A native LightGlue caller: include/lightglue_b200.h, liblightglue_b200.so and the CUDA runtime, nothing else.
//
//   nvcc -std=c++17 -I include tools/native_match_demo.cpp -L glue_factory_colon_b200/lib -llightglue_b200 \
//        -Xlinker -rpath=glue_factory_colon_b200/lib -o native_match_demo
//   ./native_match_demo DIR
//
// DIR holds
//   config.txt           "precision n_layers input_dim kdim filter_threshold B m n" (precision 1 = bf16, 2 = fp32)
//   weights/NAME.bin     one raw fp32 file per state-dict tensor, NAME = its key (LightGlue.state_dict())
//   kpts0.bin kpts1.bin desc0.bin desc1.bin    raw fp32 [B,m|n,kdim] / [B,m|n,input_dim]
//   size0.bin size1.bin (optional)             raw fp32 [B,2] (W,H)
//   counts0.bin counts1.bin (optional)         raw int32 [B] valid keypoints per pair
// and receives matches0/1.bin (int64), scores0/1.bin, log_assignment.bin (fp32 [B,m+1,n+1]) and desc_out0/1.bin
// (the last layer's descriptors, bf16 or fp32).
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <filesystem>
#include <fstream>
#include <string>
#include <vector>

#include "lightglue_b200.h"

namespace fs = std::filesystem;

static void die(const char* what, int code) {
  fprintf(stderr, "%s failed: %d (%s)\n", what, code,
          code > 0 ? cudaGetErrorString((cudaError_t)code) : lgb200_error_string(code));
  exit(1);
}
#define CHECK_LG(call) do { int rc_ = (call); if (rc_) die(#call, rc_); } while (0)
#define CHECK_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) die(#call, (int)e_); } while (0)

static std::vector<char> read_file(const fs::path& p) {
  std::ifstream f(p, std::ios::binary);
  if (!f) { fprintf(stderr, "cannot read %s\n", p.c_str()); exit(1); }
  return std::vector<char>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}

// device copy of a file (NULL if it is optional and absent)
static void* upload(const fs::path& p, bool optional = false) {
  if (optional && !fs::exists(p)) return nullptr;
  std::vector<char> h = read_file(p);
  void* d = nullptr;
  CHECK_CUDA(cudaMalloc(&d, h.size() ? h.size() : 1));
  CHECK_CUDA(cudaMemcpy(d, h.data(), h.size(), cudaMemcpyHostToDevice));
  return d;
}

static void download(const fs::path& p, const void* d, size_t bytes) {
  std::vector<char> h(bytes);
  CHECK_CUDA(cudaMemcpy(h.data(), d, bytes, cudaMemcpyDeviceToHost));
  std::ofstream(p, std::ios::binary).write(h.data(), (std::streamsize)bytes);
}

int main(int argc, char** argv) {
  if (argc != 2) { fprintf(stderr, "usage: %s DIR\n", argv[0]); return 2; }
  const fs::path dir = argv[1];
  lgb200_match_config cfg;
  int B, m, n;
  {
    std::ifstream f(dir / "config.txt");
    if (!(f >> cfg.precision >> cfg.n_layers >> cfg.input_dim >> cfg.kdim >> cfg.filter_threshold >> B >> m >> n)) {
      fprintf(stderr, "bad config.txt\n");
      return 1;
    }
  }
  CHECK_LG(lgb200_device_ok());

  // weights: every file under weights/, packed once
  std::vector<std::string> names;
  std::vector<const float*> tensors;
  for (const auto& e : fs::directory_iterator(dir / "weights")) {
    if (e.path().extension() != ".bin") continue;
    names.push_back(e.path().stem().string());
    tensors.push_back((const float*)upload(e.path()));
  }
  std::vector<const char*> cnames;
  for (const auto& s : names) cnames.push_back(s.c_str());
  int entries;
  long long pack_bytes;
  CHECK_LG(lgb200_weight_table_size(&cfg, &entries, &pack_bytes));
  void* pack = nullptr;
  CHECK_CUDA(cudaMalloc(&pack, pack_bytes));
  std::vector<const void*> table(entries);
  cudaStream_t st;
  CHECK_CUDA(cudaStreamCreate(&st));
  CHECK_LG(lgb200_pack_weights(&cfg, (int)names.size(), cnames.data(), tensors.data(), pack, pack_bytes,
                               table.data(), st));
  CHECK_CUDA(cudaStreamSynchronize(st));
  for (const float* t : tensors) CHECK_CUDA(cudaFree((void*)t));  // the pack holds everything the forward reads

  // inputs, outputs, workspace
  const float* kpts0 = (const float*)upload(dir / "kpts0.bin");
  const float* kpts1 = (const float*)upload(dir / "kpts1.bin");
  const float* desc0 = (const float*)upload(dir / "desc0.bin");
  const float* desc1 = (const float*)upload(dir / "desc1.bin");
  const float* size0 = (const float*)upload(dir / "size0.bin", true);
  const float* size1 = (const float*)upload(dir / "size1.bin", true);
  const int32_t* counts0 = (const int32_t*)upload(dir / "counts0.bin", true);
  const int32_t* counts1 = (const int32_t*)upload(dir / "counts1.bin", true);
  const size_t es = cfg.precision == LGB200_BF16 ? 2 : 4;
  const size_t n_m0 = (size_t)B * m, n_m1 = (size_t)B * n, n_la = (size_t)B * (m + 1) * (n + 1);
  void *m0, *m1, *s0, *s1, *la, *d0, *d1, *ws;
  CHECK_CUDA(cudaMalloc(&m0, n_m0 * 8 + 8));
  CHECK_CUDA(cudaMalloc(&m1, n_m1 * 8 + 8));
  CHECK_CUDA(cudaMalloc(&s0, n_m0 * 4 + 4));
  CHECK_CUDA(cudaMalloc(&s1, n_m1 * 4 + 4));
  CHECK_CUDA(cudaMalloc(&la, n_la * 4));
  CHECK_CUDA(cudaMalloc(&d0, n_m0 * 256 * es + 1));
  CHECK_CUDA(cudaMalloc(&d1, n_m1 * 256 * es + 1));
  long long ws_bytes;
  CHECK_LG(lgb200_match_workspace(&cfg, B, m, n, &ws_bytes));
  CHECK_CUDA(cudaMalloc(&ws, ws_bytes));

  CHECK_LG(lgb200_match(&cfg, table.data(), B, m, n, kpts0, kpts1, desc0, desc1, size0, size1, counts0, counts1,
                        (int64_t*)m0, (int64_t*)m1, (float*)s0, (float*)s1, (float*)la, d0, d1, ws, ws_bytes, st));
  CHECK_CUDA(cudaStreamSynchronize(st));

  download(dir / "matches0.bin", m0, n_m0 * 8);
  download(dir / "matches1.bin", m1, n_m1 * 8);
  download(dir / "scores0.bin", s0, n_m0 * 4);
  download(dir / "scores1.bin", s1, n_m1 * 4);
  download(dir / "log_assignment.bin", la, n_la * 4);
  download(dir / "desc_out0.bin", d0, n_m0 * 256 * es);
  download(dir / "desc_out1.bin", d1, n_m1 * 256 * es);
  printf("matched %d pair(s) of %d x %d keypoints\n", B, m, n);
  CHECK_CUDA(cudaStreamDestroy(st));
  return 0;
}
