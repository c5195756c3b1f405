// fa_mlp.cu -- K7: batched inference of the web app's emotion classifier on the 53-dim feature rows (SURVEY 8(f) rank 3).
//
// The reference classifies every syllable row with an ml5.js / tf.js "Sequential" of Dense layers
// (/root/reference/dist/nnmodel/<db>/cats_emotion/model.json: 53 -> 256 relu -> 64 relu -> 16 relu -> 4 softmax, float32),
// after ml5's min-max normalisation of the inputs with the ranges of model_meta.json
// (/root/reference/src/neuralmodel.js:540-585 predict_single -> classifyMultiple; vote in /root/reference/src/prediction.js:47-169).
// Here the rows are usually already on the device (the dense feature table of a finished fa_handle), so classification
// needs no PCIe round trip of the features: only 4 floats per row come back.
//
// Mapping: one CTA per tile of kRowsPerCta rows; all weights (<= ~128 KB float32) are staged once per CTA in shared memory
// by coalesced loads; activations ping-pong between two shared buffers; thread t computes output unit t of the layer for
// every row of the tile (weights read once per tile from shared memory, conflict-free: consecutive threads read consecutive
// columns).  float32 accumulation in index order with explicit fmaf -- the same DAG as the numpy-free reference loop in
// tests/ (tf.js's WebGL summation order is unspecified, so parity with the app is to 1e-5, stated in the tests).
// ~31 k MAC per row: a few microseconds per batch -- the only dense contraction near the path and far too small for
// tensor cores to matter (north_star).
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "fa_internal.cuh"

struct fa_mlp {
  int device = 0;
  int n_layers = 0;
  int dims[FA_MLP_MAX_LAYERS + 1] = {0};
  int act[FA_MLP_MAX_LAYERS] = {0};
  int w_off[FA_MLP_MAX_LAYERS] = {0}, b_off[FA_MLP_MAX_LAYERS] = {0};
  int n_params = 0, max_dim = 0;
  float* d_params = nullptr;     // kernels (row-major [in][out]) and biases, layer after layer
  double* d_norm = nullptr;      // [2][in]: min, max
  double* d_rows = nullptr;      // staging for host rows
  float* d_out = nullptr;
  size_t cap_rows = 0;
  std::string err;
};

namespace {

constexpr int kRowsPerCta = 8;
constexpr int kMlpThreads = 256;
// the activation buffers of the widest model fit the 200 KB that mlp_launch gives a CTA
static_assert(2 * kRowsPerCta * FA_MLP_MAX_UNITS * sizeof(float) <= 200 * 1024, "FA_MLP_MAX_UNITS is past K7's activation buffers");

struct MlpArgs {
  int n_layers;
  int dims[FA_MLP_MAX_LAYERS + 1];
  int act[FA_MLP_MAX_LAYERS];
  int w_off[FA_MLP_MAX_LAYERS], b_off[FA_MLP_MAX_LAYERS];
  int n_params, max_dim;
  const float* params;
  const double* norm;
  const double* rows;   // [n_rows][dims[0]] float64 (the feature table)
  int n_rows;
  float* out;           // [n_rows][dims[n_layers]]
};

// kSmemParams: all parameters staged once per CTA in shared memory (the shipped 53-256-64-16-4 model: 31 k floats); otherwise
// (53-512-512-8: 294 k floats = 1.2 MB) they are read where they are -- consecutive threads read consecutive output units of a
// kernel row, and the whole model stays in L2.  Same fmaf chain in the same order => same bits either way.
template <bool kSmemParams>
__global__ void __launch_bounds__(kMlpThreads) fa_mlp_kernel(const MlpArgs a) {
  extern __shared__ __align__(16) float smem[];
  const float* W = kSmemParams ? smem : a.params;
  float* act0 = smem + (kSmemParams ? ((a.n_params + 3) & ~3) : 0);   // [kRowsPerCta][max_dim]
  float* act1 = act0 + kRowsPerCta * a.max_dim;
  const int tid = threadIdx.x;
  if (kSmemParams)
    for (int i = tid; i < a.n_params; i += kMlpThreads) smem[i] = a.params[i];
  const int row0 = blockIdx.x * kRowsPerCta;
  const int nin = a.dims[0];
  // ml5 normalisation in double, then float32 (tf.tensor): (x - min) / (max - min)
  for (int i = tid; i < kRowsPerCta * nin; i += kMlpThreads) {
    const int r = i / nin, k = i - r * nin;
    float v = 0.f;
    if (row0 + r < a.n_rows) {
      const double x = a.rows[(size_t)(row0 + r) * nin + k];
      const double lo = a.norm[k], hi = a.norm[nin + k];
      v = (float)((x - lo) / (hi - lo));
    }
    act0[r * a.max_dim + k] = v;
  }
  __syncthreads();
  float* in = act0;
  float* outb = act1;
  for (int l = 0; l < a.n_layers; l++) {
    const int ni = a.dims[l], no = a.dims[l + 1];
    const float* Wl = W + a.w_off[l];
    const float* bl = W + a.b_off[l];
    for (int o = tid; o < no; o += kMlpThreads) {
      float acc[kRowsPerCta];
#pragma unroll
      for (int r = 0; r < kRowsPerCta; r++) acc[r] = 0.f;
      for (int k = 0; k < ni; k++) {
        const float w = kSmemParams ? Wl[k * no + o] : __ldg(Wl + k * no + o);
#pragma unroll
        for (int r = 0; r < kRowsPerCta; r++) acc[r] = fmaf(in[r * a.max_dim + k], w, acc[r]);
      }
      const float b = bl[o];
#pragma unroll
      for (int r = 0; r < kRowsPerCta; r++) {
        float v = acc[r] + b;
        if (a.act[l] == FA_MLP_RELU) v = v > 0.f ? v : (v != v ? v : 0.f);   // tf.relu keeps NaN
        else if (a.act[l] == FA_MLP_SIGMOID) v = 1.f / (1.f + expf(-v));
        outb[r * a.max_dim + o] = v;
      }
    }
    __syncthreads();
    if (a.act[l] == FA_MLP_SOFTMAX && tid < kRowsPerCta) {   // one thread per row: no <= a few classes
      float* v = outb + tid * a.max_dim;
      float mx = v[0];
      for (int o = 1; o < no; o++) mx = v[o] > mx ? v[o] : mx;
      float sum = 0.f;
      for (int o = 0; o < no; o++) { v[o] = expf(v[o] - mx); sum += v[o]; }
      for (int o = 0; o < no; o++) v[o] = v[o] / sum;
    }
    __syncthreads();
    float* t = in; in = outb; outb = t;
  }
  const int nout = a.dims[a.n_layers];
  for (int i = tid; i < kRowsPerCta * nout; i += kMlpThreads) {
    const int r = i / nout, o = i - r * nout;
    if (row0 + r < a.n_rows) a.out[(size_t)(row0 + r) * nout + o] = in[r * a.max_dim + o];
  }
}

int mlp_fail(fa_mlp* m, int code, const char* what, cudaError_t e = cudaSuccess) {
  if (m) {
    m->err = what;
    if (e != cudaSuccess) { m->err += ": "; m->err += cudaGetErrorString(e); }
  }
  return code;
}

int mlp_launch(fa_mlp* m, const double* d_rows, int n_rows, float* d_out, cudaStream_t s) {
  if (n_rows <= 0) return FA_OK;
  MlpArgs a;
  memset(&a, 0, sizeof(a));
  a.n_layers = m->n_layers;
  for (int l = 0; l <= m->n_layers; l++) a.dims[l] = m->dims[l];
  for (int l = 0; l < m->n_layers; l++) { a.act[l] = m->act[l]; a.w_off[l] = m->w_off[l]; a.b_off[l] = m->b_off[l]; }
  a.n_params = m->n_params; a.max_dim = m->max_dim; a.params = m->d_params; a.norm = m->d_norm;
  a.rows = d_rows; a.n_rows = n_rows; a.out = d_out;
  const int act_bytes = 2 * kRowsPerCta * m->max_dim * (int)sizeof(float);
  const int all_bytes = ((m->n_params + 3) & ~3) * (int)sizeof(float) + act_bytes;
  const int grid = (n_rows + kRowsPerCta - 1) / kRowsPerCta;
  cudaError_t e;
  if (all_bytes <= 200 * 1024) {
    e = cudaFuncSetAttribute(fa_mlp_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, all_bytes);
    if (e != cudaSuccess) return mlp_fail(m, FA_ERR_CUDA, "mlp shared memory", e);
    fa_mlp_kernel<true><<<grid, kMlpThreads, all_bytes, s>>>(a);
  } else {
    e = cudaFuncSetAttribute(fa_mlp_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, act_bytes);
    if (e != cudaSuccess) return mlp_fail(m, FA_ERR_CUDA, "mlp shared memory", e);
    fa_mlp_kernel<false><<<grid, kMlpThreads, act_bytes, s>>>(a);
  }
  e = cudaGetLastError();
  if (e != cudaSuccess) return mlp_fail(m, FA_ERR_CUDA, "mlp launch", e);
  return FA_OK;
}

int mlp_reserve(fa_mlp* m, size_t rows, bool need_rows) {
  if (rows <= m->cap_rows && (!need_rows || m->d_rows)) return FA_OK;
  const size_t want = std::max<size_t>(rows, 1024);
  if (m->d_rows) cudaFree(m->d_rows);
  if (m->d_out) cudaFree(m->d_out);
  m->d_rows = nullptr; m->d_out = nullptr; m->cap_rows = 0;
  cudaError_t e = cudaMalloc(&m->d_rows, want * m->dims[0] * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&m->d_out, want * m->dims[m->n_layers] * sizeof(float));
  if (e != cudaSuccess) return mlp_fail(m, FA_ERR_OUT_OF_MEMORY, "mlp buffers", e);
  m->cap_rows = want;
  return FA_OK;
}

}  // namespace

extern "C" {

int fa_mlp_create(int n_layers, const int* dims, const int* activations, const float* const* kernels,
                  const float* const* biases, const double* in_min, const double* in_max, int device, fa_mlp** out) {
  if (!out) return FA_ERR_INVALID_ARG;
  *out = nullptr;
  if (n_layers < 1 || n_layers > FA_MLP_MAX_LAYERS || !dims || !activations || !kernels || !biases || !in_min || !in_max)
    return FA_ERR_INVALID_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return FA_ERR_NO_DEVICE;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) return FA_ERR_NO_DEVICE;
  fa_mlp* m = new (std::nothrow) fa_mlp();
  if (!m) return FA_ERR_OUT_OF_MEMORY;
  m->device = device; m->n_layers = n_layers;
  int off = 0, mx = 0;
  for (int l = 0; l <= n_layers; l++) {
    if (dims[l] < 1) { delete m; return FA_ERR_INVALID_ARG; }
    // the activations of 8 rows must fit one CTA's shared memory; the parameters are staged there too when they fit (mlp_launch)
    if (dims[l] > FA_MLP_MAX_UNITS) { delete m; return FA_ERR_UNSUPPORTED; }
    m->dims[l] = dims[l];
    mx = dims[l] > mx ? dims[l] : mx;
  }
  for (int l = 0; l < n_layers; l++) {
    if (activations[l] < FA_MLP_LINEAR || activations[l] > FA_MLP_SOFTMAX || !kernels[l] || !biases[l]) { delete m; return FA_ERR_INVALID_ARG; }
    m->act[l] = activations[l];
    m->w_off[l] = off; off += dims[l] * dims[l + 1];
    m->b_off[l] = off; off += dims[l + 1];
  }
  m->n_params = off; m->max_dim = mx;
  std::vector<float> host((size_t)off);
  for (int l = 0; l < n_layers; l++) {
    memcpy(host.data() + m->w_off[l], kernels[l], sizeof(float) * (size_t)dims[l] * dims[l + 1]);
    memcpy(host.data() + m->b_off[l], biases[l], sizeof(float) * (size_t)dims[l + 1]);
  }
  std::vector<double> norm(2 * (size_t)dims[0]);
  for (int k = 0; k < dims[0]; k++) { norm[k] = in_min[k]; norm[dims[0] + k] = in_max[k]; }
  cudaSetDevice(device);
  cudaError_t e = cudaMalloc(&m->d_params, host.size() * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&m->d_norm, norm.size() * sizeof(double));
  if (e == cudaSuccess) e = cudaMemcpy(m->d_params, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(m->d_norm, norm.data(), norm.size() * sizeof(double), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { fa_mlp_destroy(m); return FA_ERR_CUDA; }
  *out = m;
  return FA_OK;
}

int fa_mlp_destroy(fa_mlp* m) {
  if (!m) return FA_OK;
  cudaSetDevice(m->device);
  if (m->d_params) cudaFree(m->d_params);
  if (m->d_norm) cudaFree(m->d_norm);
  if (m->d_rows) cudaFree(m->d_rows);
  if (m->d_out) cudaFree(m->d_out);
  delete m;
  return FA_OK;
}

const char* fa_mlp_last_error(const fa_mlp* m) { return m ? m->err.c_str() : "null model"; }

int fa_mlp_classify(fa_mlp* m, const double* rows, size_t n_rows, float* probs) {
  if (!m || (n_rows && (!rows || !probs))) return FA_ERR_INVALID_ARG;
  if (n_rows == 0) return 0;
  cudaSetDevice(m->device);
  int rc = mlp_reserve(m, n_rows, true);
  if (rc != FA_OK) return rc;
  cudaError_t e = cudaMemcpy(m->d_rows, rows, n_rows * m->dims[0] * sizeof(double), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return mlp_fail(m, FA_ERR_CUDA, "mlp H2D", e);
  rc = mlp_launch(m, m->d_rows, (int)n_rows, m->d_out, nullptr);
  if (rc != FA_OK) return rc;
  e = cudaMemcpy(probs, m->d_out, n_rows * m->dims[m->n_layers] * sizeof(float), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return mlp_fail(m, FA_ERR_CUDA, "mlp D2H", e);
  return (int)n_rows;
}

}  // extern "C"

// device-resident variant: classify the dense feature table of a finished handle (defined in fa_capi.cu, which knows fa_handle)
int fa_mlp_run_device(fa_mlp* m, const double* d_rows, int n_rows, float* probs_host, cudaStream_t s) {
  cudaSetDevice(m->device);
  int rc = mlp_reserve(m, (size_t)n_rows, false);
  if (rc != FA_OK) return rc;
  rc = mlp_launch(m, d_rows, n_rows, m->d_out, s);
  if (rc != FA_OK) return rc;
  cudaError_t e = cudaMemcpyAsync(probs_host, m->d_out, (size_t)n_rows * m->dims[m->n_layers] * sizeof(float), cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return mlp_fail(m, FA_ERR_CUDA, "mlp device run", e);
  return n_rows;
}

int fa_mlp_in_dim(const fa_mlp* m) { return m->dims[0]; }
int fa_mlp_device(const fa_mlp* m) { return m->device; }
int fa_mlp_out_dim(const fa_mlp* m) { return m->dims[m->n_layers]; }
