// block_grad.cu - layout boundary of the standalone network modules' backward (segmentation3d/_b200/blocks.py).
//
// A module's forward takes and returns NCDHW fp32 tensors (the reference modules' interface) and runs NDHWC in the
// storage type in between.  Its backward therefore starts by turning the incoming NCDHW fp32 gradient into an NDHWC
// buffer (seg3d_grad_from_ncdhw) and ends by turning the input gradient back into NCDHW fp32 (seg3d_grad_to_ncdhw).  The
// input gradient is the sum of up to three NDHWC contributions, each a channel window of its own buffer: the first
// convolution's data gradient, the residual branch's gradient, and for an up block the skip half of the concat gradient.
//
// Both are shared-memory tiled transposes of a 128-voxel x 32-channel tile: 16-byte loads/stores on the NDHWC side when
// pitch, offset and base allow them (scalar otherwise), and on the NCDHW side one warp per channel row, 32 consecutive
// fp32 voxels = 128 contiguous bytes per warp access.  Contributions are summed in fp32 in argument order g0 + g1 + g2.
#include "common.cuh"

namespace {

constexpr int BG_TV = 128;        // voxels per tile
constexpr int BG_TC = 32;         // channels per tile
constexpr int BG_THREADS = 256;

struct GradSrc {
  const void* p[3];
  int ld[3], off[3];
};

template <typename T>
__device__ __forceinline__ void load_vec(const T* p, float* v);        // 16 bytes: 16 / sizeof(T) channels
template <> __device__ __forceinline__ void load_vec<float>(const float* p, float* v) {
  const float4 q = *reinterpret_cast<const float4*>(p);
  v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
}
template <> __device__ __forceinline__ void load_vec<__half>(const __half* p, float* v) {
  Vec8<__half> q; q.load(p); q.get(v);
}
template <> __device__ __forceinline__ void load_vec<__nv_bfloat16>(const __nv_bfloat16* p, float* v) {
  Vec8<__nv_bfloat16> q; q.load(p); q.get(v);
}
template <typename T>
__device__ __forceinline__ void store_vec(T* p, const float* v);
template <> __device__ __forceinline__ void store_vec<float>(float* p, const float* v) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
template <> __device__ __forceinline__ void store_vec<__half>(__half* p, const float* v) {
  Vec8<__half> q; q.set(v); q.store(p);
}
template <> __device__ __forceinline__ void store_vec<__nv_bfloat16>(__nv_bfloat16* p, const float* v) {
  Vec8<__nv_bfloat16> q; q.set(v); q.store(p);
}

// NDHWC contributions (storage type) -> out[n][c][v] fp32.  grid (voxel tiles, channel tiles, N)
template <typename T, bool VEC>
__global__ void __launch_bounds__(BG_THREADS)
grad_to_ncdhw_kernel(GradSrc s, int nsrc, int C, long long nvox, float* __restrict__ out) {
  constexpr int V = 16 / sizeof(T);
  __shared__ float tile[BG_TC][BG_TV + 1];
  const int n = blockIdx.z, c0 = blockIdx.y * BG_TC;
  const long long v0 = (long long)blockIdx.x * BG_TV;
  const size_t row0 = (size_t)n * nvox;
  if (VEC) {
    constexpr int GPR = BG_TC / V;                     // vector groups per voxel row of the tile
    for (int i = threadIdx.x; i < BG_TV * GPR; i += BG_THREADS) {
      const int vl = i / GPR, cl = (i % GPR) * V;
      float acc[V];
#pragma unroll
      for (int j = 0; j < V; ++j) acc[j] = 0.f;
      if (v0 + vl < nvox && c0 + cl < C) {             // C % V == 0: a group is wholly inside or outside
        const size_t r = row0 + v0 + vl;
        for (int k = 0; k < nsrc; ++k) {
          float t[V];
          load_vec<T>(static_cast<const T*>(s.p[k]) + r * s.ld[k] + s.off[k] + c0 + cl, t);
#pragma unroll
          for (int j = 0; j < V; ++j) acc[j] += t[j];
        }
      }
#pragma unroll
      for (int j = 0; j < V; ++j) tile[cl + j][vl] = acc[j];
    }
  } else {
    for (int i = threadIdx.x; i < BG_TV * BG_TC; i += BG_THREADS) {
      const int vl = i / BG_TC, cl = i % BG_TC;
      float acc = 0.f;
      if (v0 + vl < nvox && c0 + cl < C) {
        const size_t r = row0 + v0 + vl;
        for (int k = 0; k < nsrc; ++k) acc += to_f32<T>(static_cast<const T*>(s.p[k])[r * s.ld[k] + s.off[k] + c0 + cl]);
      }
      tile[cl][vl] = acc;
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int r = warp; r < BG_TC * (BG_TV / 32); r += BG_THREADS / 32) {
    const int cl = r / (BG_TV / 32), vl = (r % (BG_TV / 32)) * 32 + lane;
    if (c0 + cl < C && v0 + vl < nvox) out[((size_t)n * C + c0 + cl) * nvox + v0 + vl] = tile[cl][vl];
  }
}

// in[n][c][v] fp32 -> out[(n*nvox + v)*ld + off + c] in the storage type.  grid (voxel tiles, channel tiles, N)
template <typename T, bool VEC>
__global__ void __launch_bounds__(BG_THREADS)
grad_from_ncdhw_kernel(const float* __restrict__ in, int C, long long nvox, T* __restrict__ out, int ld, int off) {
  constexpr int V = 16 / sizeof(T);
  __shared__ float tile[BG_TC][BG_TV + 1];
  const int n = blockIdx.z, c0 = blockIdx.y * BG_TC;
  const long long v0 = (long long)blockIdx.x * BG_TV;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int r = warp; r < BG_TC * (BG_TV / 32); r += BG_THREADS / 32) {
    const int cl = r / (BG_TV / 32), vl = (r % (BG_TV / 32)) * 32 + lane;
    tile[cl][vl] = (c0 + cl < C && v0 + vl < nvox) ? in[((size_t)n * C + c0 + cl) * nvox + v0 + vl] : 0.f;
  }
  __syncthreads();
  const size_t row0 = (size_t)n * nvox;
  if (VEC) {
    constexpr int GPR = BG_TC / V;
    for (int i = threadIdx.x; i < BG_TV * GPR; i += BG_THREADS) {
      const int vl = i / GPR, cl = (i % GPR) * V;
      if (v0 + vl >= nvox || c0 + cl >= C) continue;
      float t[V];
#pragma unroll
      for (int j = 0; j < V; ++j) t[j] = tile[cl + j][vl];
      store_vec<T>(out + (row0 + v0 + vl) * ld + off + c0 + cl, t);
    }
  } else {
    for (int i = threadIdx.x; i < BG_TV * BG_TC; i += BG_THREADS) {
      const int vl = i / BG_TC, cl = i % BG_TC;
      if (v0 + vl < nvox && c0 + cl < C) out[(row0 + v0 + vl) * ld + off + c0 + cl] = from_f32<T>(tile[cl][vl]);
    }
  }
}

// a 16-byte access at every (voxel, channel group) needs C, pitch and offset in whole vectors and an aligned base
bool vec_ok(const void* p, int ld, int off, int C, int elem) {
  const int v = 16 / elem;
  return C % v == 0 && ld % v == 0 && off % v == 0 && ((uintptr_t)p) % 16 == 0;
}

int elem_size(int dtype) { return dtype == SEG3D_F32 ? 4 : 2; }

}  // namespace

extern "C" int seg3d_grad_to_ncdhw(int dtype, int n_contrib, const void* g0, int ld0, int off0, const void* g1, int ld1, int off1,
                                   const void* g2, int ld2, int off2, int C, int N, int64_t nvox, float* out, void* stream) {
  SEG3D_REQUIRE(n_contrib >= 1 && n_contrib <= 3 && C > 0 && N > 0 && nvox > 0 && out, "grad_to_ncdhw: bad arguments");
  GradSrc s;
  const void* p[3] = {g0, g1, g2};
  const int ld[3] = {ld0, ld1, ld2}, off[3] = {off0, off1, off2};
  bool vec = true;
  for (int k = 0; k < 3; ++k) {
    s.p[k] = p[k]; s.ld[k] = ld[k]; s.off[k] = off[k];
    if (k >= n_contrib) continue;
    SEG3D_REQUIRE(p[k] && off[k] >= 0 && ld[k] >= off[k] + C, "grad_to_ncdhw: contribution %d: bad pointer, pitch or offset", k);
    vec = vec && vec_ok(p[k], ld[k], off[k], C, elem_size(dtype));
  }
  SEG3D_REQUIRE((nvox + BG_TV - 1) / BG_TV < (1LL << 31) && N <= 65535, "grad_to_ncdhw: too large");
  dim3 grid((unsigned)((nvox + BG_TV - 1) / BG_TV), (C + BG_TC - 1) / BG_TC, N);
  SEG3D_REQUIRE(grid.y <= 65535, "grad_to_ncdhw: C too large");
  cudaStream_t st = (cudaStream_t)stream;
  SEG3D_DISPATCH_DTYPE(dtype, T, {
    if (vec) grad_to_ncdhw_kernel<T, true><<<grid, BG_THREADS, 0, st>>>(s, n_contrib, C, nvox, out);
    else     grad_to_ncdhw_kernel<T, false><<<grid, BG_THREADS, 0, st>>>(s, n_contrib, C, nvox, out);
  });
  SEG3D_CHECK_LAUNCH("grad_to_ncdhw_kernel");
  return SEG3D_OK;
}

extern "C" int seg3d_grad_from_ncdhw(int dtype, const float* in, int C, int N, int64_t nvox, void* out, int ld, int off,
                                     void* stream) {
  SEG3D_REQUIRE(in && out && C > 0 && N > 0 && nvox > 0 && off >= 0 && ld >= off + C, "grad_from_ncdhw: bad arguments");
  SEG3D_REQUIRE((nvox + BG_TV - 1) / BG_TV < (1LL << 31) && N <= 65535, "grad_from_ncdhw: too large");
  dim3 grid((unsigned)((nvox + BG_TV - 1) / BG_TV), (C + BG_TC - 1) / BG_TC, N);
  SEG3D_REQUIRE(grid.y <= 65535, "grad_from_ncdhw: C too large");
  const bool vec = vec_ok(out, ld, off, C, elem_size(dtype));
  cudaStream_t st = (cudaStream_t)stream;
  SEG3D_DISPATCH_DTYPE(dtype, T, {
    if (vec) grad_from_ncdhw_kernel<T, true><<<grid, BG_THREADS, 0, st>>>(in, C, nvox, (T*)out, ld, off);
    else     grad_from_ncdhw_kernel<T, false><<<grid, BG_THREADS, 0, st>>>(in, C, nvox, (T*)out, ld, off);
  });
  SEG3D_CHECK_LAUNCH("grad_from_ncdhw_kernel");
  return SEG3D_OK;
}
