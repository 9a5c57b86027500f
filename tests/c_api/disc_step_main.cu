// C-only host of the discriminator's training step (no Python, no model.py): the body of train_eval_discriminator
// (deepbedmap_b200/train.py, srgan_train.py:1084-1166) on a dbm_disc handle -- zero the gradients, D([real; fake]) with
// one BatchNormalization batch per half, RaGAN loss and its logit gradients, backward, Adam.
//   usage: disc_step_main <precision: 0 = bf16, 1 = fp32> <steps k> <n> <arrays.bin> <real.bin> <fake.bin> <out.bin>
//   arrays.bin : the 60 arrays of dbm_disc_array_info, in its order, float32, concatenated (N as one float)
//   real.bin, fake.bin : (n,1,36,36) float32
//   out.bin    : k x (d_loss, d_accu), then the 60 arrays after the last step, in the order of arrays.bin
// Built and run by tests/test_gpu_disc_c_api.py.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "deepbedmap_b200.h"

#define CHECK(call)                                                          \
  do {                                                                       \
    int rc_ = (call);                                                        \
    if (rc_ != 0) {                                                          \
      fprintf(stderr, "%s failed (%d): %s\n", #call, rc_, dbm_last_error()); \
      return 1;                                                              \
    }                                                                        \
  } while (0)

#define CUDA_CHECK(call)                                                           \
  do {                                                                             \
    cudaError_t e_ = (call);                                                       \
    if (e_ != cudaSuccess) {                                                       \
      fprintf(stderr, "%s failed: %s\n", #call, cudaGetErrorString(e_));           \
      return 1;                                                                    \
    }                                                                              \
  } while (0)

static std::vector<float> read_all(const char* path) {
  FILE* f = fopen(path, "rb");
  if (!f) { fprintf(stderr, "cannot open %s\n", path); exit(2); }
  fseek(f, 0, SEEK_END);
  long bytes = ftell(f);
  fseek(f, 0, SEEK_SET);
  std::vector<float> v(bytes / 4);
  if (fread(v.data(), 4, v.size(), f) != v.size()) { fprintf(stderr, "short read of %s\n", path); exit(2); }
  fclose(f);
  return v;
}

static long array_size(int ndim, const int* dims) {
  long s = 1;
  for (int i = 0; i < ndim; ++i) s *= dims[i];
  return s;
}

int main(int argc, char** argv) {
  if (argc != 8) { fprintf(stderr, "usage: see the header of this file\n"); return 2; }
  const int precision = atoi(argv[1]), k = atoi(argv[2]), n = atoi(argv[3]);
  // Adam defaults of deepbedmap_b200.train.Adam / chainer.optimizers.Adam as the reference sets it up (:1043-1048)
  const float alpha = 1.6e-4f, beta1 = 0.9f, beta2 = 0.999f, eps = 1e-8f;
  CHECK(dbm_set_deterministic(1));
  dbm_disc* disc = nullptr;
  CHECK(dbm_disc_create(&disc));
  CHECK(dbm_disc_set_precision(disc, precision));
  const long np = dbm_disc_count_params(disc);
  const int na = dbm_disc_num_arrays(disc);
  // the optimizer owns parameters, gradients and its moments; the handle views the first two
  float *params, *grads, *m, *v;
  CUDA_CHECK(cudaMalloc(&params, np * 4));
  CUDA_CHECK(cudaMalloc(&grads, np * 4));
  CUDA_CHECK(cudaMalloc(&m, np * 4));
  CUDA_CHECK(cudaMalloc(&v, np * 4));
  CUDA_CHECK(cudaMemset(m, 0, np * 4));
  CUDA_CHECK(cudaMemset(v, 0, np * 4));
  CHECK(dbm_disc_bind_params(disc, params));
  CHECK(dbm_disc_bind_grads(disc, grads));
  std::vector<float> arrays = read_all(argv[4]);
  long pos = 0;
  for (int i = 0; i < na; ++i) {
    const char* key;
    int ndim, dims[4];
    CHECK(dbm_disc_array_info(disc, i, &key, &ndim, dims, nullptr));
    const long s = array_size(ndim, dims);
    if (pos + s > (long)arrays.size()) { fprintf(stderr, "arrays.bin is too short\n"); return 1; }
    CHECK(dbm_disc_set_param(disc, key, arrays.data() + pos, ndim, dims));
    pos += s;
  }
  if (pos != (long)arrays.size()) { fprintf(stderr, "arrays.bin holds %zu floats, expected %ld\n", arrays.size(), pos); return 1; }
  const size_t img = 36 * 36;
  std::vector<float> real = read_all(argv[5]), fake = read_all(argv[6]);
  if (real.size() != n * img || fake.size() != n * img) { fprintf(stderr, "real/fake have the wrong size\n"); return 1; }
  float *x, *logits, *dlogit, *out2;
  void* ws;
  const size_t wsb = dbm_disc_workspace_bytes(disc, 2 * n);
  CUDA_CHECK(cudaMalloc(&x, 2 * n * img * 4));
  CUDA_CHECK(cudaMalloc(&logits, 2 * n * 4));
  CUDA_CHECK(cudaMalloc(&dlogit, 2 * n * 4));
  CUDA_CHECK(cudaMalloc(&out2, 2 * 4));
  CUDA_CHECK(cudaMalloc(&ws, wsb));
  CUDA_CHECK(cudaMemcpy(x, real.data(), n * img * 4, cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMemcpy(x + n * img, fake.data(), n * img * 4, cudaMemcpyHostToDevice));
  cudaStream_t st;
  CUDA_CHECK(cudaStreamCreate(&st));
  std::vector<float> metrics(2 * k);
  for (int t = 1; t <= k; ++t) {
    CHECK(dbm_disc_zero_grads(disc, st));
    CHECK(dbm_disc_forward(disc, x, 2 * n, 2, 1, 1, logits, ws, wsb, st));
    CHECK(dbm_ragan_loss_f32(logits, logits + n, n, 1.f, 0.f, 1.f, out2, dlogit, dlogit + n, st));
    CHECK(dbm_disc_backward(disc, dlogit, ws, wsb, st));
    CHECK(dbm_adam_step_f32(params, grads, m, v, np, alpha, beta1, beta2, eps, t, 1.f, st));
    CHECK(dbm_disc_mark_updated(disc));
    CUDA_CHECK(cudaMemcpyAsync(metrics.data() + 2 * (t - 1), out2, 2 * 4, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
  }
  FILE* f = fopen(argv[7], "wb");
  if (!f) { fprintf(stderr, "cannot write %s\n", argv[7]); return 1; }
  fwrite(metrics.data(), 4, metrics.size(), f);
  for (int i = 0; i < na; ++i) {
    const char* key;
    int ndim, dims[4];
    CHECK(dbm_disc_array_info(disc, i, &key, &ndim, dims, nullptr));
    std::vector<float> a(array_size(ndim, dims));
    CHECK(dbm_disc_get_param(disc, key, a.data()));
    fwrite(a.data(), 4, a.size(), f);
  }
  fclose(f);
  CHECK(dbm_disc_destroy(disc));
  printf("ok: %d steps, n = %d, %d arrays, %ld parameters, workspace %zu bytes, %ld kernel launches\n", k, n, na, np, wsb,
         dbm_launch_count());
  return 0;
}
