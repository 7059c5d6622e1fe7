// Loss and optimizer of the training step as libgnc kernels (reference utils/train_model.py:9-10, 38-42:
// nn.CrossEntropyLoss + optim.Adam(lr=1e-3)), so that a step launches no framework arithmetic:
//   * cross entropy forward + backward over [B, C] logits in one launch (B rows, one thread each, fixed-order sum);
//   * Adam over ONE flat parameter / gradient / state buffer in one launch (the parameters of the model are views of
//     a flat buffer, utils/distributed.FlatAdam), with the data-parallel 1 / world_size folded into the gradient read.
#include "common.cuh"

namespace gnc {

// loss[0] = scale * sum_b (logsumexp(logits[b]) - logits[b, label[b]]), also added to total[0] when given;
// dlogits[b, c] = scale * (softmax - onehot)
__global__ void __launch_bounds__(256) cross_entropy_kernel(const float* __restrict__ logits, long long ld,
                                                            const long long* __restrict__ labels, int B, int C, float scale,
                                                            float* __restrict__ loss, float* __restrict__ total,
                                                            float* __restrict__ dlogits, long long ldd, int* __restrict__ bad) {
  __shared__ float part[256];
  float mine = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float* row = logits + (long long)b * ld;
    const long long lab = labels[b];
    if (lab < 0 || lab >= C) { if (bad) atomicExch(bad, 1); continue; }
    float mx = row[0];
    for (int c = 1; c < C; ++c) mx = fmaxf(mx, row[c]);
    float se = 0.f;
    for (int c = 0; c < C; ++c) se += expf(row[c] - mx);
    const float lse = mx + logf(se);
    mine += lse - row[lab];
    if (dlogits) {
      float* d = dlogits + (long long)b * ldd;
      const float inv = 1.f / se;
      for (int c = 0; c < C; ++c) d[c] = scale * (expf(row[c] - mx) * inv - (c == lab ? 1.f : 0.f));
    }
  }
  part[threadIdx.x] = mine;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < blockDim.x; ++i) s += part[i];       // fixed order: deterministic
    s *= scale;
    if (loss) loss[0] = s;
    if (total) total[0] += s;
  }
}

// torch.optim.Adam's update (amsgrad off, weight decay off), one element per thread, 128-bit accesses, with the
// roundings of its default (foreach) CUDA path, so that the parameters come out bit for bit as torch's:
//   m = fma(1 - b1, g - m, m);  v = fma(1 - b2, g g, round(v b2));  p = fma(-lr / bc1, m / (sqrt(v) / sqrt(bc2) + eps), p)
// (every other step is rounded on its own: torch runs them as separate foreach kernels)
__device__ __forceinline__ void adam_elem(float& p, float& m, float& v, float g, float one_minus_b1, float b2, float one_minus_b2,
                                          float neg_step_size, float bc2_sqrt, float eps) {
  m = __fmaf_rn(one_minus_b1, __fsub_rn(g, m), m);
  v = __fmaf_rn(one_minus_b2, __fmul_rn(g, g), __fmul_rn(v, b2));
  p = __fmaf_rn(neg_step_size, __fdiv_rn(m, __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2_sqrt), eps)), p);
}

__global__ void __launch_bounds__(256) adam_step_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                        float* __restrict__ v, long long n4, long long n, float grad_scale,
                                                        float one_minus_b1, float b2, float one_minus_b2, float neg_step_size,
                                                        float bc2_sqrt, float eps) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n4) {
    float4 pv = reinterpret_cast<float4*>(p)[i], mv = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
    const float4 gv = reinterpret_cast<const float4*>(g)[i];
    const float gs[4] = {gv.x * grad_scale, gv.y * grad_scale, gv.z * grad_scale, gv.w * grad_scale};
    float* pp = &pv.x; float* mp = &mv.x; float* vp = &vv.x;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      adam_elem(pp[c], mp[c], vp[c], gs[c], one_minus_b1, b2, one_minus_b2, neg_step_size, bc2_sqrt, eps);
    }
    reinterpret_cast<float4*>(p)[i] = pv; reinterpret_cast<float4*>(m)[i] = mv; reinterpret_cast<float4*>(v)[i] = vv;
  }
  if (i == 0) {                                                // the n % 4 tail
    for (long long j = n4 * 4; j < n; ++j) {
      adam_elem(p[j], m[j], v[j], g[j] * grad_scale, one_minus_b1, b2, one_minus_b2, neg_step_size, bc2_sqrt, eps);
    }
  }
}

}  // namespace gnc

using namespace gnc;

extern "C" {

int gnc_cross_entropy_f32(const float* logits, int64_t ld, const int64_t* labels, int B, int C, float scale, float* loss,
                          float* total, float* dlogits, int64_t ldd, int* bad_label_flag, gnc_stream_t stream) {
  GNC_REQUIRE(logits && labels && (loss || total) && B >= 0 && C >= 1 && ld >= C && (!dlogits || ldd >= C), "cross_entropy: bad arguments");
  cross_entropy_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(logits, ld, reinterpret_cast<const long long*>(labels), B, C, scale,
                                                            loss, total, dlogits, ldd, bad_label_flag);
  return check_launch("cross_entropy_kernel");
}

int gnc_adam_step_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, double lr, double beta1,
                      double beta2, double eps, int64_t step, float grad_scale, gnc_stream_t stream) {
  GNC_REQUIRE(param && grad && exp_avg && exp_avg_sq && n >= 0 && step >= 1, "adam_step: bad arguments");
  GNC_REQUIRE(aligned16(param) && aligned16(grad) && aligned16(exp_avg) && aligned16(exp_avg_sq), "adam_step: 16-byte aligned buffers");
  if (n == 0) return GNC_OK;
  // bias corrections in double on the host, as torch's scalar path computes them
  // (hyper-parameters arrive as doubles: torch forms 1 - beta in double before rounding to float, and
  // 1 - float(0.999) differs from float(1 - 0.999) by 1.3e-5 relative)
  const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
  const float neg_step_size = (float)(-(lr / bc1));
  const float bc2_sqrt = (float)pow(bc2, 0.5);
  const long long n4 = n / 4;
  long long blocks = ceil_div<long long>(n4 > 0 ? n4 : 1, 256);
  adam_step_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, n4, n, grad_scale,
                                                                       (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), neg_step_size,
                                                                       bc2_sqrt, (float)eps);
  return check_launch("adam_step_kernel");
}

int gnc_zero_f32(float* buf, int64_t n, gnc_stream_t stream) {
  GNC_REQUIRE(buf && n >= 0, "zero: bad arguments");
  cudaError_t e = cudaMemsetAsync(buf, 0, (size_t)n * sizeof(float), (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(GNC_ECUDA, "zero: cudaMemsetAsync: %s", cudaGetErrorString(e));
  return GNC_OK;
}

}  // extern "C"
