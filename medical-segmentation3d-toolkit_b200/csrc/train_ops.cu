// train_ops.cu - the parameter side of the training step (reference core/seg_train.py:83,119-127):
//   seg3d_gather_pack : table-driven strided gather with a cast - ONE launch re-packs every convolution weight of the network
//                       from the reference's fp32 OIDHW / IODHW parameters into the kernels' layouts (tensor-core [tap][Cout][Cin]
//                       in the storage type, SIMT [tap][Cin][Cout], split hi/lo halves, the folded narrow-output layout, the
//                       flipped / transposed data-gradient weights), and one more launch turns the kernel-layout weight
//                       gradients back into parameter layout;
//   seg3d_adam_step   : torch.optim.Adam's update (the reference's optimiser, lr / betas / eps / weight decay) over one flat
//                       fp32 range holding every parameter of the network;
//   seg3d_adam_step_ranges : the same update over a list of sub-ranges, each with its own step count (parameters without a
//                       gradient are left out of the list and keep their values and moments, as torch.optim.Adam skips them).
// Both are pure streaming kernels over ~58 MB; they replace ~250 tiny framework launches per step.
#include "common.cuh"

namespace {

__device__ __forceinline__ void store_as(void* dst, long long i, int dtype, float v) {
  if (dtype == SEG3D_F32) reinterpret_cast<float*>(dst)[i] = v;
  else if (dtype == SEG3D_F16) reinterpret_cast<__half*>(dst)[i] = __float2half_rn(v);
  else reinterpret_cast<__nv_bfloat16*>(dst)[i] = __float2bfloat16_rn(v);
}

// Block b serves chunk block_map[2b+1] (SEG3D_PACK_CHUNK elements) of entry block_map[2b]: the entries range from 2 to 1.8 M
// elements, and a (chunks x entries) grid would launch ~100 000 empty blocks.  Index arithmetic is 32-bit (an entry has
// < 2^31 elements); consecutive threads take consecutive DESTINATION elements, so stores coalesce and the gathers hit L2 (all
// parameters together are 58 MB).
__global__ void __launch_bounds__(256)
gather_pack_kernel(const seg3d_pack_entry* __restrict__ table, const int32_t* __restrict__ block_map) {
  __shared__ seg3d_pack_entry se;
  if (threadIdx.x == 0) se = table[block_map[2 * blockIdx.x]];
  __syncthreads();
  const uint32_t first = (uint32_t)block_map[2 * blockIdx.x + 1] * (uint32_t)SEG3D_PACK_CHUNK;
  const uint32_t s1 = (uint32_t)se.size[1], s2 = (uint32_t)se.size[2], s3 = (uint32_t)se.size[3], s4 = (uint32_t)se.size[4];
  const uint32_t total = (uint32_t)se.size[0] * s1 * s2 * s3 * s4;
  const uint32_t n = total - first < (uint32_t)SEG3D_PACK_CHUNK ? total : first + (uint32_t)SEG3D_PACK_CHUNK;
  const float* __restrict__ src = se.src;
  for (uint32_t i = first + threadIdx.x; i < n; i += blockDim.x) {
    uint32_t r = i;
    const uint32_t i4 = r % s4; r /= s4;
    const uint32_t i3 = r % s3; r /= s3;
    const uint32_t i2 = r % s2; r /= s2;
    const uint32_t i1 = r % s1; const uint32_t i0 = r / s1;
    const bool inside = (int)i0 < se.limit[0] && (int)i1 < se.limit[1] && (int)i2 < se.limit[2] && (int)i3 < se.limit[3] && (int)i4 < se.limit[4];
    const long long so = se.src_base + (long long)i0 * se.src_stride[0] + (long long)i1 * se.src_stride[1] + (long long)i2 * se.src_stride[2] +
                         (long long)i3 * se.src_stride[3] + (long long)i4 * se.src_stride[4];
    const long long d_o = se.dst_base + (long long)i0 * se.dst_stride[0] + (long long)i1 * se.dst_stride[1] + (long long)i2 * se.dst_stride[2] +
                          (long long)i3 * se.dst_stride[3] + (long long)i4 * se.dst_stride[4];
    float v = inside ? src[so] : 0.f;
    if (se.kind != SEG3D_PACK_PLAIN) {             // split operands: hi = f16(w), lo = f16(w - hi)
      const float hi = __half2float(__float2half_rn(v));
      v = se.kind == SEG3D_PACK_SPLIT_HI ? hi : v - hi;
    }
    store_as(se.dst, d_o, se.dtype, v);
  }
}

// torch/optim/adam.py::_single_tensor_adam (no amsgrad, no maximize):
//   g += wd * p;  m.lerp_(g, 1 - b1);  v = b2 * v + (1 - b2) * g * g;  p -= step_size * m / (sqrt(v) / sqrt(bc2) + eps)
// over elements [0, n) of one range, element i taken by thread `first` + k * `stride` of the grid
__device__ __forceinline__ void adam_range(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                           float* __restrict__ v, long long n, float b1, float b2, float eps, float wd,
                                           float step_size, float bc2_sqrt, long long first, long long stride) {
  const long long n4 = n >> 2;
  for (long long i = first; i < n4; i += stride) {
    float4 pp = reinterpret_cast<float4*>(p)[i], gg = reinterpret_cast<const float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
    float* pa = &pp.x; float* ga = &gg.x; float* ma = &mm.x; float* va = &vv.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float gr = wd != 0.f ? fmaf(wd, pa[j], ga[j]) : ga[j];
      ma[j] = ma[j] + (1.f - b1) * (gr - ma[j]);
      va[j] = fmaf(1.f - b2, gr * gr, b2 * va[j]);
      pa[j] -= step_size * (ma[j] / (sqrtf(va[j]) / bc2_sqrt + eps));
    }
    reinterpret_cast<float4*>(p)[i] = pp; reinterpret_cast<float4*>(m)[i] = mm; reinterpret_cast<float4*>(v)[i] = vv;
  }
  for (long long i = (n4 << 2) + first; i < n; i += stride) {
    const float gr = wd != 0.f ? fmaf(wd, p[i], g[i]) : g[i];
    const float mi = m[i] + (1.f - b1) * (gr - m[i]);
    const float vi = fmaf(1.f - b2, gr * gr, b2 * v[i]);
    m[i] = mi; v[i] = vi;
    p[i] -= step_size * (mi / (sqrtf(vi) / bc2_sqrt + eps));
  }
}

__global__ void __launch_bounds__(256)
adam_step_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
                 float b1, float b2, float eps, float wd, float step_size, float bc2_sqrt) {
  adam_range(p, g, m, v, n, b1, b2, eps, wd, step_size, bc2_sqrt, (long long)blockIdx.x * blockDim.x + threadIdx.x,
             (long long)gridDim.x * blockDim.x);
}

// seg3d_adam_step_ranges: up to ADAM_RANGES_PER_LAUNCH ranges per launch, passed by value; blockIdx.y picks the range
constexpr int ADAM_RANGES_PER_LAUNCH = 32;
struct AdamRanges {
  long long off[ADAM_RANGES_PER_LAUNCH], n[ADAM_RANGES_PER_LAUNCH];
  float step_size[ADAM_RANGES_PER_LAUNCH], bc2_sqrt[ADAM_RANGES_PER_LAUNCH];
};

__global__ void __launch_bounds__(256)
adam_ranges_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                   const AdamRanges r, float b1, float b2, float eps, float wd) {
  const int k = blockIdx.y;
  const long long o = r.off[k];
  adam_range(p + o, g + o, m + o, v + o, r.n[k], b1, b2, eps, wd, r.step_size[k], r.bc2_sqrt[k],
             (long long)blockIdx.x * blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x);
}

// the bias corrections of one step count, in double as torch computes them, rounded once to fp32
void adam_corrections(float lr, float beta1, float beta2, long long step, float& step_size, float& bc2_sqrt) {
  const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
  step_size = (float)((double)lr / bc1);
  bc2_sqrt = (float)sqrt(bc2);
}

}  // namespace

extern "C" int seg3d_gather_pack(const seg3d_pack_entry* table, const int32_t* block_map, int n_blocks, void* stream) {
  SEG3D_REQUIRE(table && block_map && n_blocks > 0, "gather_pack: bad arguments");
  gather_pack_kernel<<<n_blocks, 256, 0, (cudaStream_t)stream>>>(table, block_map);
  SEG3D_CHECK_LAUNCH("gather_pack_kernel");
  return SEG3D_OK;
}

extern "C" int seg3d_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                               float lr, float beta1, float beta2, float eps, float weight_decay, int step, void* stream) {
  SEG3D_REQUIRE(param && grad && exp_avg && exp_avg_sq && n > 0 && step >= 1, "adam_step: bad arguments");
  SEG3D_REQUIRE(((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) % 16 == 0, "adam_step: pointers must be 16-byte aligned");
  float step_size, bc2_sqrt;
  adam_corrections(lr, beta1, beta2, step, step_size, bc2_sqrt);
  long long want = ((n >> 2) + 255) / 256;
  const int cap = 8 * seg3d_num_sms();
  const int gx = (int)(want < 1 ? 1 : (want > cap ? cap : want));
  adam_step_kernel<<<gx, 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, n, beta1, beta2, eps, weight_decay, step_size, bc2_sqrt);
  SEG3D_CHECK_LAUNCH("adam_step_kernel");
  return SEG3D_OK;
}

extern "C" int seg3d_adam_step_ranges(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                                      const seg3d_adam_range* ranges, int n_ranges, float lr, float beta1, float beta2,
                                      float eps, float weight_decay, void* stream) {
  SEG3D_REQUIRE(param && grad && exp_avg && exp_avg_sq && ranges && n_ranges > 0, "adam_step_ranges: bad arguments");
  SEG3D_REQUIRE(((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) % 16 == 0,
                "adam_step_ranges: pointers must be 16-byte aligned");
  const int cap = 8 * seg3d_num_sms();
  for (int r0 = 0; r0 < n_ranges; r0 += ADAM_RANGES_PER_LAUNCH) {
    const int nr = n_ranges - r0 < ADAM_RANGES_PER_LAUNCH ? n_ranges - r0 : ADAM_RANGES_PER_LAUNCH;
    AdamRanges t;
    long long longest = 0;
    for (int k = 0; k < nr; ++k) {
      const seg3d_adam_range& e = ranges[r0 + k];
      SEG3D_REQUIRE(e.offset >= 0 && e.offset % 4 == 0 && e.n > 0 && e.step >= 1,
                    "adam_step_ranges: range %d needs offset >= 0 (a multiple of 4), n > 0 and step >= 1", r0 + k);
      t.off[k] = e.offset; t.n[k] = e.n;
      adam_corrections(lr, beta1, beta2, e.step, t.step_size[k], t.bc2_sqrt[k]);
      longest = e.n > longest ? e.n : longest;
    }
    const long long want = ((longest >> 2) + 255) / 256;
    const int per = (cap + nr - 1) / nr;
    const int gx = (int)(want < 1 ? 1 : (want > per ? per : want));
    adam_ranges_kernel<<<dim3(gx, nr), 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, t, beta1, beta2, eps, weight_decay);
    SEG3D_CHECK_LAUNCH("adam_ranges_kernel");
  }
  return SEG3D_OK;
}
