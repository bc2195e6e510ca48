// cin1_dgrad.cu - data gradient of the single-channel input block (in_block.conv, k3 s1 p1, 1 -> 16 channels):
//   dx[n][z][y][x] = sum over taps (a, b, c) and channels co of w[a][b][c][co] * gy[n][z+1-a][y+1-b][x+1-c][co]
// with zero padding, accumulated in fp32 and written as fp32 straight into the NCDHW [N,1,D,H,W] input gradient.
//
// The work is 27 x 16 FMAs per voxel (6 GFLOP per 8 x 96^3 step), so a SIMT kernel moving 16 gy channels in and one fp32
// value out per voxel suffices.  A block owns an 8 x 32 (y, x) column and marches a chunk of ZC planes in z: each gy plane
// (with its one-voxel y/x halo) is staged once in shared memory as fp32 [channel][position] and feeds the three output
// planes it touches (z = p-1, p, p+1) through three rolling accumulators per thread, so a staged value is read once per
// in-plane tap instead of three times.
#include "common.cuh"

namespace {

constexpr int DG_TY = 8, DG_TX = 32, DG_ZC = 16;
constexpr int DG_HY = DG_TY + 2, DG_HX = DG_TX + 2, DG_HP = DG_HY * DG_HX;   // 340 halo positions per plane
constexpr int DG_THREADS = DG_TY * DG_TX;

template <typename T>
__device__ __forceinline__ void load16(const T* p, float* v) {
  if constexpr (sizeof(T) == 4) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 q = reinterpret_cast<const float4*>(p)[i];
      v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
    }
  } else {
    Vec8<T> a, b;
    a.load(p); b.load(p + 8);
    a.get(v); b.get(v + 8);
  }
}

template <typename T>
__global__ void __launch_bounds__(DG_THREADS)
cin1_dgrad_kernel(const T* __restrict__ gy, int ld, const float* __restrict__ w, float* __restrict__ dx,
                  int D, int H, int W, int nzc) {
  __shared__ float sg[16][DG_HP];
  __shared__ float4 sw[27 * 4];                    // w[tap][16] as 4 float4 per tap
  const int tid = threadIdx.x, tx = tid % DG_TX, ty = tid / DG_TX;
  const int x0 = blockIdx.x * DG_TX, y0 = blockIdx.y * DG_TY;
  const int n = blockIdx.z / nzc, z0 = (blockIdx.z % nzc) * DG_ZC;
  const int z1 = min(z0 + DG_ZC, D);
  if (tid < 27 * 4) sw[tid] = reinterpret_cast<const float4*>(w)[tid];
  const size_t plane = (size_t)H * W;
  const T* gyn = gy + (size_t)n * D * plane * ld;
  float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f;       // output planes p-1, p, p+1
  for (int p = z0 - 1; p <= z1; ++p) {
    const bool live = p >= 0 && p < D;
    if (live) {
      __syncthreads();                              // the previous plane's readers are done
      for (int i = tid; i < DG_HP; i += DG_THREADS) {
        const int yy = y0 - 1 + i / DG_HX, xx = x0 - 1 + i % DG_HX;
        float v[16];
        if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
          load16(gyn + ((size_t)p * plane + (size_t)yy * W + xx) * ld, v);
        } else {
#pragma unroll
          for (int c = 0; c < 16; ++c) v[c] = 0.f;
        }
#pragma unroll
        for (int c = 0; c < 16; ++c) sg[c][i] = v[c];
      }
      __syncthreads();
      // gy at in-plane offset (1-b, 1-c) feeds tap (a, b, c) of output plane p + a - 1
#pragma unroll
      for (int b = 0; b < 3; ++b) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int pos = (ty + 2 - b) * DG_HX + (tx + 2 - c);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 w0 = sw[((0 * 3 + b) * 3 + c) * 4 + q];
            const float4 w1 = sw[((1 * 3 + b) * 3 + c) * 4 + q];
            const float4 w2 = sw[((2 * 3 + b) * 3 + c) * 4 + q];
            const float g0 = sg[4 * q][pos], g1 = sg[4 * q + 1][pos], g2 = sg[4 * q + 2][pos], g3 = sg[4 * q + 3][pos];
            acc0 = fmaf(w0.x, g0, acc0); acc0 = fmaf(w0.y, g1, acc0); acc0 = fmaf(w0.z, g2, acc0); acc0 = fmaf(w0.w, g3, acc0);
            acc1 = fmaf(w1.x, g0, acc1); acc1 = fmaf(w1.y, g1, acc1); acc1 = fmaf(w1.z, g2, acc1); acc1 = fmaf(w1.w, g3, acc1);
            acc2 = fmaf(w2.x, g0, acc2); acc2 = fmaf(w2.y, g1, acc2); acc2 = fmaf(w2.z, g2, acc2); acc2 = fmaf(w2.w, g3, acc2);
          }
        }
      }
    }
    // output plane p-1 has seen all three of its gy planes
    const int zo = p - 1, yo = y0 + ty, xo = x0 + tx;
    if (zo >= z0 && zo < z1 && yo < H && xo < W) dx[((size_t)n * D + zo) * plane + (size_t)yo * W + xo] = acc0;
    acc0 = acc1; acc1 = acc2; acc2 = 0.f;
  }
}

}  // namespace

extern "C" int seg3d_conv3d_cin1_dgrad(int dtype, const void* gy, int ld, const float* w, float* dx,
                                       int N, int D, int H, int W, void* stream) {
  SEG3D_REQUIRE(gy && w && dx && N > 0 && D > 0 && H > 0 && W > 0, "conv3d_cin1_dgrad: bad arguments");
  const int esz = dtype == SEG3D_F32 ? 4 : 2;
  SEG3D_REQUIRE(ld >= 16 && (ld * esz) % 16 == 0, "conv3d_cin1_dgrad: gy pitch must be >= 16 channels and a multiple of 16 bytes");
  SEG3D_REQUIRE(((uintptr_t)gy) % 16 == 0 && ((uintptr_t)w) % 16 == 0, "conv3d_cin1_dgrad: gy and w must be 16-byte aligned");
  const int nzc = (D + DG_ZC - 1) / DG_ZC;
  SEG3D_REQUIRE((long long)N * nzc < 65536 && (H + DG_TY - 1) / DG_TY < 65536, "conv3d_cin1_dgrad: grid too large");
  const dim3 grid((W + DG_TX - 1) / DG_TX, (H + DG_TY - 1) / DG_TY, N * nzc);
  cudaStream_t st = (cudaStream_t)stream;
  SEG3D_DISPATCH_DTYPE(dtype, T,
    cin1_dgrad_kernel<T><<<grid, DG_THREADS, 0, st>>>(reinterpret_cast<const T*>(gy), ld, w, dx, D, H, W, nzc));
  SEG3D_CHECK_LAUNCH("cin1_dgrad_kernel");
  return SEG3D_OK;
}
