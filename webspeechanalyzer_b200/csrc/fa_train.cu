// fa_train.cu -- K9: training of the web app's feature-row classifier (a Sequential of Dense layers, softmax output,
// categorical cross-entropy) on the GPU, many independent jobs per launch.
//
// The web app trains this net in the browser with ml5 (src/neuralmodel.js train_nn); ml5 / tf.js seed nothing, so the
// algorithm here is builder-defined and stated in DESIGN.md "K9": Glorot-uniform start values drawn by the host, ml5's
// min-max normalisation (double, then float32, exactly as K7), a seeded Feistel order of each epoch (include/fa_train.h),
// mini-batches whose last one averages over its own rows, and SGD or Adam (tf.js constants) in float32.
//
// Mapping: one CTA of kTrainThreads threads per job, and one launch for the whole run -- a step is a few microseconds of
// arithmetic with a strict dependency on the previous one, so the host never comes between steps.  Parameters, gradients
// and Adam moments of a job live in global memory (they stay in L1 / L2: 124 KB for 53-256-64-16-4, 1.2 MB for
// 53-512-512-8); the activations of a batch ([rows][dims[l]] per layer) live in shared memory when they fit and in a
// per-job global scratch otherwise (same code, same order, same bits).  The backward sweep overwrites each layer's
// activations with its deltas in place.  Per step: the batch's rows and inputs, one phase per layer forward (thread =
// output unit x 8 rows in registers), softmax / loss / output delta (thread = row), per layer a gradient phase
// (thread = parameter, rows in order) and a delta phase (thread = input unit x 8 rows), then the optimizer over all
// parameters; __syncthreads between phases.  float32 with explicit fmaf in a fixed index order (--fmad=false), loss and
// accuracy summed by one thread in row order: a job's result depends on nothing but its own inputs.  Jobs fill the SMs.
// No tensor cores: ~31 k MAC per row and step-to-step dependency, not FLOPs, bound the run.
//
// ptxas (sm_100a, -Xptxas -v, CUDA 12.9): fa_train_kernel 64 registers, 16 bytes static shared memory, 0 bytes stack,
// 0 bytes spill stores / loads; dynamic shared memory 9.5 KB + the activations (50 KB for 53-256-64-16-4 at batch 32,
// 139 KB for 53-512-512-8 at batch 32).
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "fa_internal.cuh"
#include "fa_train.h"

namespace {

constexpr int kTrainThreads = 512;
constexpr int kTile = 8;                  // rows per thread in the forward and delta phases (register tile)
constexpr int kSmemCap = 200 * 1024;      // dynamic shared memory a job may take
constexpr float kBeta1 = 0.9f, kBeta2 = 0.999f, kOneMinusBeta1 = 0.1f, kOneMinusBeta2 = 0.001f, kEpsilon = 1e-7f;

struct TrainArgs {
  int n_layers;
  int dims[FA_MLP_MAX_LAYERS + 1];
  int act[FA_MLP_MAX_LAYERS];
  int w_off[FA_MLP_MAX_LAYERS], b_off[FA_MLP_MAX_LAYERS];
  int a_off[FA_MLP_MAX_LAYERS + 1];      // activations (then deltas) of layer l: [bpad][dims[l]] floats at a_off[l]
  int n_params, n_act, act_smem_off;     // act_smem_off: byte offset of the activations in shared memory (act_g == nullptr)
  int batch, bpad, epochs, optimizer, given_ranges;
  float lr;
  const double* rows;                    // [n_rows][dims[0]]
  const int* labels;                     // [n_rows]
  const long long* job_off;              // [J + 1]
  const int* row_idx;
  const unsigned long long* seeds;       // [J]
  float* params;                         // [J][n_params]: start values in, trained values out
  float* grad;                           // [J][n_params]
  float* m1; float* m2;                  // [J][n_params] Adam moments (zero at the start), nullptr for SGD
  float* act_g;                          // [J][n_act] when the activations do not fit shared memory, else nullptr
  double* ranges;                        // [J][2][dims[0]]: given ranges in (given_ranges), the ranges used out
  double* history;                       // [J][epochs][2]: mean loss, accuracy
  int* bad_row;                          // [J]: a table row with a non-finite value (INT_MAX: none)
};

__global__ void __launch_bounds__(kTrainThreads) fa_train_kernel(const TrainArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_bad;
  const int j = blockIdx.x, tid = threadIdx.x;
  const int L = a.n_layers, d0 = a.dims[0], nout = a.dims[L], bpad = a.bpad;
  double* red = reinterpret_cast<double*>(smem_raw);     // [2][kTrainThreads] partial min / max
  double* rng = red + 2 * kTrainThreads;                  // [2][d0] min, max
  double* loss_r = rng + 2 * d0;                          // [bpad]
  int* rowid = reinterpret_cast<int*>(loss_r + bpad);     // [bpad]
  int* lab = rowid + bpad;
  int* hit_r = lab + bpad;
  float* A = a.act_g ? a.act_g + (size_t)j * a.n_act : reinterpret_cast<float*>(smem_raw + a.act_smem_off);
  float* P = a.params + (size_t)j * a.n_params;
  float* G = a.grad + (size_t)j * a.n_params;
  float* M1 = a.m1 ? a.m1 + (size_t)j * a.n_params : nullptr;
  float* M2 = a.m2 ? a.m2 + (size_t)j * a.n_params : nullptr;
  double* R = a.ranges + (size_t)j * 2 * d0;
  const int* list = a.row_idx + a.job_off[j];
  const int n = (int)(a.job_off[j + 1] - a.job_off[j]);
  const unsigned long long seed = a.seeds[j];

  // ---- input ranges over the job's rows (min / max: exact in any order) and the non-finite check ----
  if (tid == 0) s_bad = INT_MAX;
  const int C = d0 < kTrainThreads ? d0 : kTrainThreads;   // columns at a time
  const int groups = kTrainThreads / C;                    // threads per column
  for (int c0 = 0; c0 < d0; c0 += C) {
    __syncthreads();
    const int g = tid / C, c = c0 + tid % C;
    double lo = INFINITY, hi = -INFINITY;
    if (g < groups && c < d0) {
      for (int i = g; i < n; i += groups) {
        const int row = list[i];
        const double x = a.rows[(size_t)row * d0 + c];
        if (!isfinite(x)) atomicMin(&s_bad, row);
        lo = fmin(lo, x);
        hi = fmax(hi, x);
      }
    }
    red[tid] = lo;
    red[kTrainThreads + tid] = hi;
    __syncthreads();
    if (tid < C && c < d0) {
      for (int k = 1; k < groups; k++) {
        lo = fmin(lo, red[k * C + tid]);
        hi = fmax(hi, red[kTrainThreads + k * C + tid]);
      }
      if (a.given_ranges) {
        lo = R[c];
        hi = R[d0 + c];
      } else if (hi == lo) {
        hi = lo + 1.0;                                     // a constant column maps to 0, in training and in K7
      }
      rng[c] = lo;
      rng[d0 + c] = hi;
      R[c] = lo;
      R[d0 + c] = hi;
    }
  }
  __syncthreads();
  if (s_bad != INT_MAX) {
    if (tid == 0) a.bad_row[j] = s_bad;
    return;
  }

  float acc_b1 = 1.f, acc_b2 = 1.f;                        // beta^t as float32 running products (tf.js)
  for (int e = 0; e < a.epochs; e++) {
    double loss_sum = 0.0;
    long long hits = 0;
    for (int s0 = 0; s0 < n; s0 += a.batch) {
      const int bc = n - s0 < a.batch ? n - s0 : a.batch;
      for (int r = tid; r < bpad; r += kTrainThreads) {
        const int row = r < bc ? list[fa_perm((uint32_t)(s0 + r), (uint32_t)n, seed, (uint32_t)e)] : -1;
        rowid[r] = row;
        lab[r] = row >= 0 ? a.labels[row] : 0;
      }
      __syncthreads();
      // ml5 normalisation in double, then float32; padding rows are zero
      for (int i = tid; i < bpad * d0; i += kTrainThreads) {
        const int r = i / d0, c = i - r * d0;
        float v = 0.f;
        if (r < bc) v = (float)((a.rows[(size_t)rowid[r] * d0 + c] - rng[c]) / (rng[d0 + c] - rng[c]));
        A[i] = v;
      }
      __syncthreads();

      // ---- forward ----
      for (int l = 0; l < L; l++) {
        const int ni = a.dims[l], no = a.dims[l + 1], act = a.act[l];
        const float* W = P + a.w_off[l];
        const float* b = P + a.b_off[l];
        const float* in = A + a.a_off[l];
        float* out = A + a.a_off[l + 1];
        for (int it = tid; it < (bpad / kTile) * no; it += kTrainThreads) {
          const int rg = it / no, o = it - rg * no;
          const float* x = in + rg * kTile * ni;
          float acc[kTile];
#pragma unroll
          for (int r = 0; r < kTile; r++) acc[r] = 0.f;
          for (int k = 0; k < ni; k++) {
            const float w = W[k * no + o];
#pragma unroll
            for (int r = 0; r < kTile; r++) acc[r] = fmaf(x[r * ni + k], w, acc[r]);
          }
          const float bo = b[o];
#pragma unroll
          for (int r = 0; r < kTile; r++) {
            float v = acc[r] + bo;
            if (act == FA_MLP_RELU) v = v > 0.f ? v : (v != v ? v : 0.f);
            else if (act == FA_MLP_SIGMOID) v = 1.f / (1.f + expf(-v));
            out[(rg * kTile + r) * no + o] = v;
          }
        }
        __syncthreads();
      }
      // ---- softmax (K7's), loss, arg-max and the output delta (p - onehot) / rows, one thread per row ----
      for (int r = tid; r < bpad; r += kTrainThreads) {
        float* v = A + a.a_off[L] + r * nout;
        if (r < bc) {
          float mx = v[0];
          for (int o = 1; o < nout; o++) mx = v[o] > mx ? v[o] : mx;
          float sum = 0.f;
          for (int o = 0; o < nout; o++) { v[o] = expf(v[o] - mx); sum += v[o]; }
          int best = 0;
          for (int o = 0; o < nout; o++) {
            v[o] = v[o] / sum;
            if (v[o] > v[best]) best = o;
          }
          const int y = lab[r];
          loss_r[r] = -log(fmax((double)v[y], 1e-7));
          hit_r[r] = best == y;
          for (int o = 0; o < nout; o++) v[o] = (v[o] - (o == y ? 1.f : 0.f)) / (float)bc;
        } else {
          for (int o = 0; o < nout; o++) v[o] = 0.f;
        }
      }
      __syncthreads();
      if (tid == 0)
        for (int r = 0; r < bc; r++) { loss_sum += loss_r[r]; hits += hit_r[r]; }

      // ---- backward: gradients with the step's weights, deltas in place of the activations ----
      for (int l = L - 1; l >= 0; l--) {
        const int ni = a.dims[l], no = a.dims[l + 1];
        const float* W = P + a.w_off[l];
        float* in = A + a.a_off[l];
        const float* dz = A + a.a_off[l + 1];
        float* Gl = G + a.w_off[l];                        // kernel [ni][no], then the bias (b_off = w_off + ni * no)
        for (int it = tid; it < ni * no + no; it += kTrainThreads) {
          float g = 0.f;
          if (it < ni * no) {
            const int k = it / no, o = it - k * no;
            for (int r = 0; r < bc; r++) g = fmaf(in[r * ni + k], dz[r * no + o], g);
          } else {
            const int o = it - ni * no;
            for (int r = 0; r < bc; r++) g += dz[r * no + o];
          }
          Gl[it] = g;
        }
        __syncthreads();
        if (l == 0) break;
        const int act = a.act[l - 1];
        for (int it = tid; it < (bpad / kTile) * ni; it += kTrainThreads) {
          const int rg = it / ni, k = it - rg * ni;
          const float* d = dz + rg * kTile * no;
          float acc[kTile];
#pragma unroll
          for (int r = 0; r < kTile; r++) acc[r] = 0.f;
          for (int o = 0; o < no; o++) {
            const float w = W[k * no + o];
#pragma unroll
            for (int r = 0; r < kTile; r++) acc[r] = fmaf(d[r * no + o], w, acc[r]);
          }
#pragma unroll
          for (int r = 0; r < kTile; r++) {
            float* y = in + (rg * kTile + r) * ni + k;
            if (act == FA_MLP_RELU) *y = *y > 0.f ? acc[r] : 0.f;
            else if (act == FA_MLP_SIGMOID) *y = acc[r] * (*y * (1.f - *y));
            else *y = acc[r];
          }
        }
        __syncthreads();
      }

      // ---- optimizer; a zero step leaves a parameter's bits as they are ----
      if (a.optimizer == FA_OPT_ADAM) {
        acc_b1 *= kBeta1;
        acc_b2 *= kBeta2;
        const float c1 = 1.f - acc_b1, c2 = 1.f - acc_b2;
        for (int p = tid; p < a.n_params; p += kTrainThreads) {
          const float g = G[p];
          const float m = kBeta1 * M1[p] + kOneMinusBeta1 * g;
          const float v = kBeta2 * M2[p] + kOneMinusBeta2 * (g * g);
          M1[p] = m;
          M2[p] = v;
          const float u = a.lr * ((m / c1) / (sqrtf(v / c2) + kEpsilon));
          if (u != 0.f) P[p] = P[p] - u;
        }
      } else {
        for (int p = tid; p < a.n_params; p += kTrainThreads) {
          const float u = a.lr * G[p];
          if (u != 0.f) P[p] = P[p] - u;
        }
      }
      __syncthreads();
    }
    if (tid == 0) {
      a.history[((size_t)j * a.epochs + e) * 2] = loss_sum / n;
      a.history[((size_t)j * a.epochs + e) * 2 + 1] = (double)hits / n;
    }
  }
}

// device buffers of one fa_mlp_train call, freed on every return path
struct DeviceBuffers {
  std::vector<void*> ptrs;
  cudaError_t err = cudaSuccess;
  template <class T>
  T* alloc(size_t count) {
    void* p = nullptr;
    if (err == cudaSuccess) err = cudaMalloc(&p, (count ? count : 1) * sizeof(T));
    if (p) ptrs.push_back(p);
    return static_cast<T*>(p);
  }
  template <class T>
  T* upload(const T* src, size_t count) {
    T* d = alloc<T>(count);
    if (err == cudaSuccess && count) err = cudaMemcpy(d, src, count * sizeof(T), cudaMemcpyHostToDevice);
    return d;
  }
  ~DeviceBuffers() {
    for (void* p : ptrs) cudaFree(p);
  }
};

}  // namespace

extern "C" int fa_mlp_train(int n_layers, const int* dims, const int* activations, const double* rows, size_t n_rows,
                            const int32_t* labels, int n_jobs, const int64_t* job_offsets, const int32_t* row_idx,
                            const uint64_t* seeds, const float* init_params, const double* in_ranges,
                            const fa_train_opts* opts, int device, float* out_params, double* out_ranges,
                            double* out_history, char* err, size_t err_cap) {
  if (err && err_cap) err[0] = 0;
  auto fail = [&](int code, const char* fmt, long long x = 0, long long y = 0, long long z = 0) {
    if (err && err_cap) snprintf(err, err_cap, fmt, x, y, z);
    return code;
  };
  if (n_layers < 1 || n_layers > FA_MLP_MAX_LAYERS) return fail(FA_ERR_INVALID_ARG, "n_layers must be in [1, %lld]", FA_MLP_MAX_LAYERS);
  if (!dims || !activations || !opts || !job_offsets || !row_idx || !seeds || !init_params || !out_params || !out_ranges ||
      (!out_history && opts->epochs > 0) || (n_rows && (!rows || !labels)))
    return fail(FA_ERR_INVALID_ARG, "null argument");
  for (int l = 0; l <= n_layers; l++)
    if (dims[l] < 1 || dims[l] > 4096) return fail(FA_ERR_INVALID_ARG, "dims[%lld] must be in [1, 4096]", l);
  for (int l = 0; l + 1 < n_layers; l++)
    if (activations[l] != FA_MLP_LINEAR && activations[l] != FA_MLP_RELU && activations[l] != FA_MLP_SIGMOID)
      return fail(FA_ERR_INVALID_ARG, "hidden layer %lld: the activation must be linear, relu or sigmoid", l);
  if (activations[n_layers - 1] != FA_MLP_SOFTMAX) return fail(FA_ERR_INVALID_ARG, "the output activation must be softmax");
  if (opts->batch_size < 1 || opts->batch_size > 65536) return fail(FA_ERR_INVALID_ARG, "batch_size must be in [1, 65536]");
  if (opts->epochs < 0) return fail(FA_ERR_INVALID_ARG, "epochs must be >= 0");
  if (opts->optimizer != FA_OPT_SGD && opts->optimizer != FA_OPT_ADAM) return fail(FA_ERR_INVALID_ARG, "unknown optimizer");
  if (!std::isfinite(opts->learning_rate)) return fail(FA_ERR_INVALID_ARG, "learning_rate must be finite");
  if (n_jobs < 1 || job_offsets[0] != 0) return fail(FA_ERR_INVALID_ARG, "n_jobs must be >= 1 and job_offsets[0] must be 0");
  const int nout = dims[n_layers];
  for (int j = 0; j < n_jobs; j++) {
    if (job_offsets[j + 1] <= job_offsets[j]) return fail(FA_ERR_INVALID_ARG, "job %lld is empty", j);
    if (job_offsets[j + 1] - job_offsets[j] > INT_MAX) return fail(FA_ERR_INVALID_ARG, "job %lld has more than 2^31 - 1 rows", j);
  }
  const long long n_idx = job_offsets[n_jobs];
  for (long long i = 0; i < n_idx; i++) {
    const int32_t r = row_idx[i];
    if (r < 0 || (size_t)r >= n_rows) return fail(FA_ERR_INVALID_ARG, "row index %lld at position %lld is outside [0, n_rows)", r, i);
    if (labels[r] < 0 || labels[r] >= nout)
      return fail(FA_ERR_INVALID_ARG, "label %lld of row %lld is outside [0, %lld)", labels[r], r, nout);
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev)
    return fail(FA_ERR_NO_DEVICE, "no CUDA device");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10)
    return fail(FA_ERR_NO_DEVICE, "not an sm_100 device");
  cudaSetDevice(device);

  TrainArgs a;
  memset(&a, 0, sizeof(a));
  a.n_layers = n_layers;
  int off = 0, act_floats = 0;
  a.bpad = (opts->batch_size + kTile - 1) / kTile * kTile;
  for (int l = 0; l <= n_layers; l++) {
    a.dims[l] = dims[l];
    a.a_off[l] = act_floats;
    act_floats += a.bpad * dims[l];
  }
  for (int l = 0; l < n_layers; l++) {
    a.act[l] = activations[l];
    a.w_off[l] = off; off += dims[l] * dims[l + 1];
    a.b_off[l] = off; off += dims[l + 1];
  }
  a.n_params = off;
  a.n_act = act_floats;
  a.batch = opts->batch_size;
  a.epochs = opts->epochs;
  a.optimizer = opts->optimizer;
  a.lr = (float)opts->learning_rate;
  a.given_ranges = in_ranges != nullptr;
  const int d0 = dims[0];
  const size_t J = (size_t)n_jobs, P = (size_t)a.n_params;
  const int fixed = ((2 * kTrainThreads + 2 * d0 + a.bpad) * (int)sizeof(double) + 3 * a.bpad * (int)sizeof(int) + 15) & ~15;
  const bool act_smem = fixed + act_floats * (int)sizeof(float) <= kSmemCap;
  const int smem = act_smem ? fixed + act_floats * (int)sizeof(float) : fixed;
  a.act_smem_off = fixed;

  DeviceBuffers buf;
  a.rows = buf.upload(rows, n_rows * d0);
  a.labels = buf.upload(reinterpret_cast<const int*>(labels), n_rows);
  a.job_off = buf.upload(reinterpret_cast<const long long*>(job_offsets), J + 1);
  a.row_idx = buf.upload(reinterpret_cast<const int*>(row_idx), (size_t)n_idx);
  a.seeds = buf.upload(reinterpret_cast<const unsigned long long*>(seeds), J);
  a.params = buf.upload(init_params, J * P);
  a.grad = buf.alloc<float>(J * P);
  if (a.optimizer == FA_OPT_ADAM) {
    a.m1 = buf.alloc<float>(J * P);
    a.m2 = buf.alloc<float>(J * P);
    if (buf.err == cudaSuccess) buf.err = cudaMemset(a.m1, 0, J * P * sizeof(float));
    if (buf.err == cudaSuccess) buf.err = cudaMemset(a.m2, 0, J * P * sizeof(float));
  }
  if (!act_smem) a.act_g = buf.alloc<float>(J * (size_t)act_floats);
  a.ranges = in_ranges ? buf.upload(in_ranges, J * 2 * d0) : buf.alloc<double>(J * 2 * d0);
  a.history = buf.alloc<double>(J * (size_t)a.epochs * 2);
  std::vector<int> bad(J, INT_MAX);
  a.bad_row = buf.upload(bad.data(), J);
  if (buf.err != cudaSuccess)
    return fail(buf.err == cudaErrorMemoryAllocation ? FA_ERR_OUT_OF_MEMORY : FA_ERR_CUDA, "device buffers");

  cudaError_t e = cudaFuncSetAttribute(fa_train_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e == cudaSuccess) {
    fa_train_kernel<<<n_jobs, kTrainThreads, smem>>>(a);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(bad.data(), a.bad_row, J * sizeof(int), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) {
    if (err && err_cap) snprintf(err, err_cap, "training kernel: %s", cudaGetErrorString(e));
    return FA_ERR_CUDA;
  }
  for (size_t j = 0; j < J; j++)
    if (bad[j] != INT_MAX) return fail(FA_ERR_INVALID_ARG, "row %lld has a non-finite value", bad[j]);
  e = cudaMemcpy(out_params, a.params, J * P * sizeof(float), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(out_ranges, a.ranges, J * 2 * d0 * sizeof(double), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && a.epochs)
    e = cudaMemcpy(out_history, a.history, J * (size_t)a.epochs * 2 * sizeof(double), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) {
    if (err && err_cap) snprintf(err, err_cap, "copy back: %s", cudaGetErrorString(e));
    return FA_ERR_CUDA;
  }
  return FA_OK;
}
