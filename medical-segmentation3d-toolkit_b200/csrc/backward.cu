// backward.cu - training-side kernels: GroupNorm(1,C)+ReLU(+residual) backward, weight gradients,
// and the backward of the output-block tail (softmax <- GN2 <- 1x1x1 conv <- ReLU <- GN1).
//
// Data-gradient (dgrad) of the convolutions needs no kernel of its own: k3 s1 p1 dgrad is the same
// convolution with flipped/transposed weights, k2s2 dgrad is the transposed conv and vice versa, so the
// forward kernels (tensor-core or SIMT) are reused through seg3d_conv3d_fwd.
//
// Unit being differentiated (conv_gn_relu3.py:16-20, residual_block3.py:24):
//     y = conv(x)                       raw, saved
//     z = gamma*(y-mean)*rstd + beta    xhat = (y-mean)*rstd
//     out = relu(z [+ res])             saved (its sign is the ReLU mask)
// Given g = dL/d out (sum of up to three contributions), dz = g*[out>0] and
// (units without a residual: the mask is recomputed as fma(y, rstd*gamma, beta - mean*rstd*gamma) > 0, the very expression
// the forward apply evaluated on the same stored y, so `out` is not read at all - a third of pass 0's traffic)
//     dy = rstd*(gamma*dz - mean_all(gamma*dz) - xhat*mean_all(gamma*dz*xhat)),
//     dgamma_c = sum dz*xhat, dbeta_c = sum dz, dres = dz, dbias_c = sum dy.
// A unit without the ReLU (a standalone ConvGnRelu3(..., do_act=False) ends in a plain GroupNorm) takes the same two passes
// with dz = g (NOACT: no mask, neither `out` nor beta read).
#include "common.cuh"

namespace {

constexpr int GN_BWD_MAXC = 512;
constexpr int GN_BWD_U = 4;

// PASS 0: per-sample sums S1 = sum gamma*dz, S2 = sum gamma*dz*xhat; per-channel dgamma, dbeta.
// PASS 1: dy (+ optional dres), per-channel dbias.
template <typename T, int PASS, bool REMASK, bool NOACT = false>
__global__ void __launch_bounds__(256, 2)
gn_bwd_kernel(const T* __restrict__ g0, int ld0, const T* __restrict__ g1, int ld1, const T* __restrict__ g2, int ld2,
              const T* __restrict__ out, int out_ld, const T* __restrict__ y, int y_ld, int C,
              const double* __restrict__ stats, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
              double* __restrict__ sums, float* __restrict__ dgamma, float* __restrict__ dbeta,
              T* __restrict__ dy, int dy_ld, T* __restrict__ dres, int dres_ld, float* __restrict__ dbias, long long nvox) {
  __shared__ float sacc[2 * GN_BWD_MAXC];
  __shared__ float red[64];
  const int n = blockIdx.y;
  float mean, rstd;
  gn_mean_rstd(stats + 2 * n, (double)nvox * C, eps, mean, rstd);
  for (int c = threadIdx.x; c < 2 * C; c += blockDim.x) sacc[c] = 0.f;
  float m1 = 0.f, m2 = 0.f;
  if (PASS == 1) {
    const double cnt = (double)nvox * C;
    m1 = (float)(sums[2 * n] / cnt); m2 = (float)(sums[2 * n + 1] / cnt);
  }
  __syncthreads();
  const int cv = C >> 3;
  // blockDim (256) is a multiple of cv and so is the grid stride: a thread keeps one channel group
  const int grp = threadIdx.x % cv, c0 = grp << 3;
  const long long vstep = (long long)gridDim.x * (blockDim.x / cv);
  float gam[8], za[8], zb[8];          // REMASK: z = fma(y, za, zb) exactly as gn_apply_kernel forms it
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    gam[j] = gamma[c0 + j];
    za[j] = rstd * gam[j];
    zb[j] = REMASK ? beta[c0 + j] - mean * za[j] : 0.f;
  }
  float a0[8], a1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { a0[j] = 0.f; a1[j] = 0.f; }
  float s1 = 0.f, s2 = 0.f;
  const size_t nb = (size_t)n * nvox;
  // GN_BWD_U voxels per iteration with every load issued before the first use: the kernel is a pure HBM stream and
  // needs ~100 KB of loads in flight per SM
  for (long long v = (long long)blockIdx.x * (blockDim.x / cv) + threadIdx.x / cv; v < nvox; v += GN_BWD_U * vstep) {
    Vec8<T> rg0[GN_BWD_U], rg1[GN_BWD_U], rg2[GN_BWD_U], ro[GN_BWD_U], ry[GN_BWD_U];
#pragma unroll
    for (int u = 0; u < GN_BWD_U; ++u) {
      const long long vu = v + u * vstep;
      const size_t vv = nb + (vu < nvox ? vu : v);           // clamp: the duplicate is masked below
      rg0[u].load(g0 + vv * ld0 + c0);
      if (g1) rg1[u].load(g1 + vv * ld1 + c0); else rg1[u].zero();
      if (g2) rg2[u].load(g2 + vv * ld2 + c0); else rg2[u].zero();
      if (!REMASK && !NOACT) ro[u].load(out + vv * out_ld + c0);
      ry[u].load(y + vv * y_ld + c0);
    }
#pragma unroll
    for (int u = 0; u < GN_BWD_U; ++u) {
      const long long vu = v + u * vstep;
      if (vu >= nvox) break;
      const size_t vv = nb + vu;
      float ga[8], gb[8], gc[8], o[8], yy[8];
      rg0[u].get(ga); rg1[u].get(gb); rg2[u].get(gc); ry[u].get(yy);
      if (!REMASK && !NOACT) ro[u].get(o);
      float dyv[8], dzv[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const bool on = NOACT || (REMASK ? (fmaf(yy[j], za[j], zb[j]) > 0.f) : (o[j] > 0.f));
        const float dz = on ? (ga[j] + gb[j] + gc[j]) : 0.f;
        const float xh = (yy[j] - mean) * rstd;
        if (PASS == 0) {
          a0[j] = fmaf(dz, xh, a0[j]); a1[j] += dz;        // the per-sample sums follow from these at the end (a block = one sample)
        } else {
          const float d = rstd * (gam[j] * dz - m1 - xh * m2);
          dyv[j] = d; dzv[j] = dz; a0[j] += d;
        }
      }
      if (PASS == 1) {
        Vec8<T> w; w.set(dyv); w.store(dy + vv * dy_ld + c0);
        if (dres) { w.set(dzv); w.store(dres + vv * dres_ld + c0); }
      }
    }
  }
  if (PASS == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) { s1 = fmaf(gam[j], a1[j], s1); s2 = fmaf(gam[j], a0[j], s2); }
  }
  // per-channel partials: lanes that own the same channel group (lane % cv) are folded with shuffles first, then
  // one shared-memory atomic per warp and channel, then one global atomic per channel per block
  for (int off = 16; off >= cv; off >>= 1) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      a0[j] += __shfl_xor_sync(0xffffffffu, a0[j], off);
      if (PASS == 0) a1[j] += __shfl_xor_sync(0xffffffffu, a1[j], off);
    }
  }
  if ((threadIdx.x & 31) < cv) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      atomicAdd(&sacc[c0 + j], a0[j]);
      if (PASS == 0) atomicAdd(&sacc[C + c0 + j], a1[j]);
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    if (PASS == 0) { atomicAdd(dgamma + c, sacc[c]); atomicAdd(dbeta + c, sacc[C + c]); }
    else if (dbias) atomicAdd(dbias + c, sacc[c]);
  }
  if (PASS == 0) block_stats_atomic(s1, s2, sums + 2 * n, red);
}

// ---- weight gradient: dW[tap][ci][co] += sum_v x[v (+) tap][ci] * dy[v][co]  (fp32, split over voxels) ------
struct WgradGeom {
  int mode, N, D, H, W;       // x spatial dims (conv input)
  int Do, Ho, Wo;             // iteration space of v (dy dims for K3/K2S2/K1; x dims for T2S2)
  int Cin, Cout, x_ld, dy_ld;
  int vps, chunk, nchunks;    // voxels per sample of the iteration space; voxels per CTA
};

template <typename T>
__global__ void __launch_bounds__(256)
wgrad_simt_kernel(const WgradGeom g, const T* __restrict__ x, const T* __restrict__ dy, float* __restrict__ dw) {
  constexpr int BM = 64, BN = 64, BK = 16;
  __shared__ __align__(16) float As[BK][BM + 4];   // x rows    [voxel][ci]
  __shared__ __align__(16) float Bs[BK][BN + 4];   // dy rows   [voxel][co]
  const int tap = blockIdx.y;
  const int tiles_n = (g.Cout + BN - 1) / BN;
  const int ci0 = (blockIdx.z / tiles_n) * BM, co0 = (blockIdx.z % tiles_n) * BN;
  const int n = blockIdx.x / g.nchunks;
  const int v_begin = (blockIdx.x % g.nchunks) * g.chunk;
  const int v_end = min(v_begin + g.chunk, g.vps);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  // loader role: 16 voxels x 64 channels per operand = 1024 elements, 4 per thread: voxel = tid/16, channels (tid%16)*4..+3
  const int lv = tid >> 4, lc = (tid & 15) * 4;
  const T* xn = x + (size_t)n * g.D * g.H * g.W * g.x_ld;
  for (int v0 = v_begin; v0 < v_end; v0 += BK) {
    const int v = v0 + lv;
    float a[4] = {0.f, 0.f, 0.f, 0.f}, b[4] = {0.f, 0.f, 0.f, 0.f};
    if (v < v_end) {
      const int vx = v % g.Wo; const int t = v / g.Wo; const int vy = t % g.Ho, vz = t / g.Ho;
      int xz, xy, xx, ok = 1; size_t dyv;
      if (g.mode == SEG3D_CONV_K3) {
        xz = vz + tap / 9 - 1; xy = vy + (tap / 3) % 3 - 1; xx = vx + tap % 3 - 1;
        ok = (xz >= 0) & (xz < g.D) & (xy >= 0) & (xy < g.H) & (xx >= 0) & (xx < g.W);
        dyv = (size_t)n * g.vps + v;
      } else if (g.mode == SEG3D_CONV_K2S2) {
        xz = 2 * vz + (tap >> 2); xy = 2 * vy + ((tap >> 1) & 1); xx = 2 * vx + (tap & 1);
        dyv = (size_t)n * g.vps + v;
      } else if (g.mode == SEG3D_CONV_T2S2) {      // v runs over x voxels; dy voxel = 2v + tap
        xz = vz; xy = vy; xx = vx;
        dyv = (((size_t)n * 2 * g.D + 2 * vz + (tap >> 2)) * 2 * g.H + 2 * vy + ((tap >> 1) & 1)) * 2 * g.W + 2 * vx + (tap & 1);
      } else { xz = vz; xy = vy; xx = vx; dyv = (size_t)n * g.vps + v; }
      if (ok) {
        const T* xp = xn + ((size_t)(xz * g.H + xy) * g.W + xx) * g.x_ld;
#pragma unroll
        for (int j = 0; j < 4; ++j) if (ci0 + lc + j < g.Cin) a[j] = to_f32<T>(xp[ci0 + lc + j]);
      }
      const T* dp = dy + dyv * g.dy_ld;
#pragma unroll
      for (int j = 0; j < 4; ++j) if (co0 + lc + j < g.Cout) b[j] = to_f32<T>(dp[co0 + lc + j]);
    }
    *reinterpret_cast<float4*>(&As[lv][lc]) = make_float4(a[0], a[1], a[2], a[3]);
    *reinterpret_cast<float4*>(&Bs[lv][lc]) = make_float4(b[0], b[1], b[2], b[3]);
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float aa[4] = {av.x, av.y, av.z, av.w}, bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
  // dw layout: K3/K2S2/K1 [tap][Cin][Cout]; T2S2 [Cin][8*Cout] (column = tap*Cout + co)
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int ci = ci0 + ty * 4 + i;
    if (ci >= g.Cin) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int co = co0 + tx * 4 + j;
      if (co >= g.Cout) continue;
      const size_t o = g.mode == SEG3D_CONV_T2S2 ? ((size_t)ci * 8 + tap) * g.Cout + co : ((size_t)tap * g.Cin + ci) * g.Cout + co;
      atomicAdd(dw + o, acc[i][j]);
    }
  }
}

// ---- output-block tail backward ------------------------------------------------------------------
// PASS 0: dl (softmax bwd) -> GN2 sums + dgamma2/dbeta2.   PASS 1: dz2 -> dW2, db2, dh -> dg1 -> GN1 sums + dgamma1/dbeta1.
// PASS 2: dy1 = GN1 backward -> store, db1.
struct TailBwdArgs {
  const double *stats1, *stats2;
  const float *gamma1, *beta1, *w2, *bias2, *gamma2, *beta2;
  const float* dprobs;            // [N][C][nvox]
  double *sums2, *sums1;          // [N][2]
  float *dgamma2, *dbeta2, *dw2, *db2, *dgamma1, *dbeta1, *db1;
  float eps;
};

template <typename T, int C, int PASS>
__global__ void __launch_bounds__(256)
tail_bwd_kernel(const T* __restrict__ y1, int ld, TailBwdArgs a, T* __restrict__ dy1, int dy_ld, long long nvox) {
  __shared__ float sw2[C * C], sb2[C], sa1[C], sb1[C], sa2[C], sbb2[C], sg1[C], sg2[C];
  __shared__ float sred[C * C + 4 * C + 4];
  const int n = blockIdx.y;
  float mean1, rstd1, mean2, rstd2;
  gn_mean_rstd(a.stats1 + 2 * n, (double)nvox * C, a.eps, mean1, rstd1);
  gn_mean_rstd(a.stats2 + 2 * n, (double)nvox * C, a.eps, mean2, rstd2);
  if (threadIdx.x < C * C) sw2[threadIdx.x] = a.w2[threadIdx.x];
  if (threadIdx.x < C) {
    const int c = threadIdx.x;
    sg1[c] = a.gamma1[c]; sg2[c] = a.gamma2[c];
    sa1[c] = rstd1 * sg1[c]; sb1[c] = a.beta1[c] - mean1 * sa1[c];
    sa2[c] = rstd2 * sg2[c]; sbb2[c] = a.beta2[c] - mean2 * sa2[c];
    sb2[c] = a.bias2 ? a.bias2[c] : 0.f;
  }
  for (int i = threadIdx.x; i < C * C + 4 * C + 4; i += blockDim.x) sred[i] = 0.f;
  __syncthreads();
  const double cnt = (double)nvox * C;
  float m1 = 0.f, m2 = 0.f, t1 = 0.f, t2 = 0.f;
  if (PASS >= 1) { m1 = (float)(a.sums2[2 * n] / cnt); m2 = (float)(a.sums2[2 * n + 1] / cnt); }
  if (PASS == 2) { t1 = (float)(a.sums1[2 * n] / cnt); t2 = (float)(a.sums1[2 * n + 1] / cnt); }

  float accA[C], accB[C], accW[C * C], accD[C];
#pragma unroll
  for (int c = 0; c < C; ++c) { accA[c] = 0.f; accB[c] = 0.f; accD[c] = 0.f; }
#pragma unroll
  for (int i = 0; i < C * C; ++i) accW[i] = 0.f;
  float s1 = 0.f, s2 = 0.f;
  const T* yn = y1 + (size_t)n * nvox * ld;
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < nvox; v += (long long)gridDim.x * blockDim.x) {
    float xh1[C], h[C], z[C], xh2[C], p[C], dl[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const float yv = to_f32<T>(yn[v * ld + c]);
      xh1[c] = (yv - mean1) * rstd1;
      h[c] = fmaxf(fmaf(yv, sa1[c], sb1[c]), 0.f);
    }
    float mx = -INFINITY;
#pragma unroll
    for (int o = 0; o < C; ++o) {
      float t = sb2[o];
#pragma unroll
      for (int c = 0; c < C; ++c) t = fmaf(sw2[o * C + c], h[c], t);
      z[o] = t; xh2[o] = (t - mean2) * rstd2;
      p[o] = fmaf(t, sa2[o], sbb2[o]); mx = fmaxf(mx, p[o]);
    }
    float den = 0.f;
#pragma unroll
    for (int o = 0; o < C; ++o) { p[o] = expf(p[o] - mx); den += p[o]; }
    const float inv = 1.f / den;
    float dot = 0.f;
#pragma unroll
    for (int o = 0; o < C; ++o) { p[o] *= inv; dl[o] = a.dprobs[((size_t)n * C + o) * nvox + v]; dot += p[o] * dl[o]; }
#pragma unroll
    for (int o = 0; o < C; ++o) dl[o] = p[o] * (dl[o] - dot);          // softmax backward
    if (PASS == 0) {
#pragma unroll
      for (int o = 0; o < C; ++o) { s1 += sg2[o] * dl[o]; s2 += sg2[o] * dl[o] * xh2[o]; accA[o] += dl[o] * xh2[o]; accB[o] += dl[o]; }
      continue;
    }
    float dz2[C], dg1[C];
#pragma unroll
    for (int o = 0; o < C; ++o) dz2[o] = rstd2 * (sg2[o] * dl[o] - m1 - xh2[o] * m2);
#pragma unroll
    for (int c = 0; c < C; ++c) {
      float t = 0.f;
#pragma unroll
      for (int o = 0; o < C; ++o) t = fmaf(sw2[o * C + c], dz2[o], t);
      dg1[c] = h[c] > 0.f ? t : 0.f;
    }
    if (PASS == 1) {
#pragma unroll
      for (int o = 0; o < C; ++o) {
        accD[o] += dz2[o];
#pragma unroll
        for (int c = 0; c < C; ++c) accW[o * C + c] += dz2[o] * h[c];
      }
#pragma unroll
      for (int c = 0; c < C; ++c) { s1 += sg1[c] * dg1[c]; s2 += sg1[c] * dg1[c] * xh1[c]; accA[c] += dg1[c] * xh1[c]; accB[c] += dg1[c]; }
    } else {
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float d = rstd1 * (sg1[c] * dg1[c] - t1 - xh1[c] * t2);
        accD[c] += d;
        dy1[((size_t)n * nvox + v) * dy_ld + c] = from_f32<T>(d);
      }
    }
  }
  // block reduction through shared atomics, then global atomics
  // warp-level sums first to keep shared atomics few
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const float va = warp_sum(accA[c]), vb = warp_sum(accB[c]), vd = warp_sum(accD[c]);
    if ((threadIdx.x & 31) == 0) { atomicAdd(&sred[c], va); atomicAdd(&sred[C + c], vb); atomicAdd(&sred[2 * C + c], vd); }
  }
  if (PASS == 1) {
#pragma unroll
    for (int i = 0; i < C * C; ++i) {
      const float vw = warp_sum(accW[i]);
      if ((threadIdx.x & 31) == 0) atomicAdd(&sred[4 * C + 4 + i], vw);
    }
  }
  {
    const float v1 = warp_sum(s1), v2 = warp_sum(s2);
    if ((threadIdx.x & 31) == 0) { atomicAdd(&sred[3 * C], v1); atomicAdd(&sred[3 * C + 1], v2); }
  }
  __syncthreads();
  if (threadIdx.x < C) {
    const int c = threadIdx.x;
    if (PASS == 0) { atomicAdd(a.dgamma2 + c, sred[c]); atomicAdd(a.dbeta2 + c, sred[C + c]); }
    if (PASS == 1) { atomicAdd(a.dgamma1 + c, sred[c]); atomicAdd(a.dbeta1 + c, sred[C + c]); atomicAdd(a.db2 + c, sred[2 * C + c]); }
    if (PASS == 2) atomicAdd(a.db1 + c, sred[2 * C + c]);
  }
  if (PASS == 1 && threadIdx.x < C * C) atomicAdd(a.dw2 + threadIdx.x, sred[4 * C + 4 + threadIdx.x]);
  if (threadIdx.x == 0) {
    if (PASS == 0) { atomicAdd(a.sums2 + 2 * n, (double)sred[3 * C]); atomicAdd(a.sums2 + 2 * n + 1, (double)sred[3 * C + 1]); }
    if (PASS == 1) { atomicAdd(a.sums1 + 2 * n, (double)sred[3 * C]); atomicAdd(a.sums1 + 2 * n + 1, (double)sred[3 * C + 1]); }
  }
}

template <typename T, int PASS>
int launch_tail_bwd(int C, dim3 grid, cudaStream_t st, const T* y1, int ld, const TailBwdArgs& a, T* dy1, int dy_ld, long long nvox) {
#define TB_CASE(CC) case CC: tail_bwd_kernel<T, CC, PASS><<<grid, 256, 0, st>>>(y1, ld, a, dy1, dy_ld, nvox); break;
  switch (C) {
    TB_CASE(1) TB_CASE(2) TB_CASE(3) TB_CASE(4) TB_CASE(5) TB_CASE(6) TB_CASE(7) TB_CASE(8)
    TB_CASE(9) TB_CASE(10) TB_CASE(11) TB_CASE(12) TB_CASE(13) TB_CASE(14) TB_CASE(15) TB_CASE(16)
    default: seg3d_set_error("tail backward: C=%d not in 1..16", C); return SEG3D_EUNSUPPORTED;
  }
#undef TB_CASE
  SEG3D_CHECK_LAUNCH("tail_bwd_kernel");
  return SEG3D_OK;
}


// ---- weight gradient of the input block (Cin == 1, Cout == 16): dW[tap][co] = sum_v x[v + tap] * dy[v][co] --------
// Register-tiled: a thread owns one (x,y) column of an 8 x 8 x 12 voxel tile and four output channels, keeps its
// 27 x 4 partial sums in registers, marches along z with the 3 x 9 input window in registers (9 shared-memory reads
// per voxel) and reads its 4 dy channels straight from global memory (a warp covers 8 consecutive voxels x 32 B).
// 108 independent FMAs per voxel per thread; the partial sums are folded once per block (shuffles, shared atomics,
// 432 global atomics).
constexpr int WC1_LZ = 12;
template <typename T>
__global__ void __launch_bounds__(256)
wgrad_cin1_kernel(const T* __restrict__ x, const T* __restrict__ dy, int dy_ld, float* __restrict__ dw,
                  int N, int D, int H, int W, int ntx, int nty, int ntz) {
  __shared__ float xs[WC1_LZ + 2][10][10];
  __shared__ float red[27 * 16];
  const int tid = threadIdx.x;
  const int q = tid & 3, vox = tid >> 2, lx = vox & 7, ly = vox >> 3;
  float acc[27][4];
#pragma unroll
  for (int t = 0; t < 27; ++t)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[t][c] = 0.f;
  for (int i = tid; i < 27 * 16; i += blockDim.x) red[i] = 0.f;
  const long long ntiles = (long long)ntx * nty * ntz * N;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    long long t = tile;
    const int x0 = (int)(t % ntx) * 8; t /= ntx;
    const int y0 = (int)(t % nty) * 8; t /= nty;
    const int z0 = (int)(t % ntz) * WC1_LZ; const int n = (int)(t / ntz);
    const T* xn = x + (size_t)n * D * H * W;
    __syncthreads();
    for (int i = tid; i < (WC1_LZ + 2) * 100; i += blockDim.x) {
      const int hx = i % 10, hy = (i / 10) % 10, hz = i / 100;
      const int gx = x0 + hx - 1, gy = y0 + hy - 1, gz = z0 + hz - 1;
      float v = 0.f;
      if (gx >= 0 && gx < W && gy >= 0 && gy < H && gz >= 0 && gz < D) v = to_f32<T>(xn[((size_t)gz * H + gy) * W + gx]);
      xs[hz][hy][hx] = v;
    }
    __syncthreads();
    const int gx = x0 + lx, gy = y0 + ly;
    const bool inplane = gx < W && gy < H;
    const T* dcol = dy + ((((size_t)n * D + z0) * H + gy) * W + gx) * dy_ld + q * 4;
    const size_t zstride = (size_t)H * W * dy_ld;
    float win[3][9];
#pragma unroll
    for (int i = 0; i < 9; ++i) { win[0][i] = xs[0][ly + i / 3][lx + i % 3]; win[1][i] = xs[1][ly + i / 3][lx + i % 3]; }
    // dy is read three z steps ahead as raw bits (converted at use: one block per SM, nothing else hides the latency)
    struct Raw { uint4 v; };
    auto load_dy = [&](int z, Raw& r) {
      r.v = make_uint4(0u, 0u, 0u, 0u);
      if (inplane && z < WC1_LZ && z0 + z < D) {
        if (sizeof(T) == 2) { const uint2 t2 = *reinterpret_cast<const uint2*>(dcol + (size_t)z * zstride); r.v.x = t2.x; r.v.y = t2.y; }
        else r.v = *reinterpret_cast<const uint4*>(dcol + (size_t)z * zstride);
      }
    };
    Raw dq[3];
    load_dy(0, dq[0]); load_dy(1, dq[1]); load_dy(2, dq[2]);
    for (int zl = 0; zl < WC1_LZ; zl += 3) {
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const int z = zl + j;
#pragma unroll
        for (int i = 0; i < 9; ++i) win[(j + 2) % 3][i] = xs[z + 2][ly + i / 3][lx + i % 3];
        float d[4];
        {
          const T* h = reinterpret_cast<const T*>(&dq[j].v);
#pragma unroll
          for (int c = 0; c < 4; ++c) d[c] = to_f32<T>(h[c]);
        }
        load_dy(z + 3, dq[j]);
#pragma unroll
        for (int kd = 0; kd < 3; ++kd)
#pragma unroll
          for (int i = 0; i < 9; ++i) {
            const float xv = win[(j + kd) % 3][i];
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[kd * 9 + i][c] = fmaf(xv, d[c], acc[kd * 9 + i][c]);
          }
      }
    }
  }
  // fold: lanes with the same channel quad (lane & 3), then warps through shared memory, then one atomic per weight
#pragma unroll
  for (int t = 0; t < 27; ++t)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float v = acc[t][c];
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      if ((tid & 31) < 4) atomicAdd(&red[t * 16 + q * 4 + c], v);
    }
  __syncthreads();
  for (int i = tid; i < 27 * 16; i += blockDim.x) atomicAdd(dw + i, red[i]);
}

}  // namespace

extern "C" int seg3d_gn_bwd(int dtype, int pass, const void* g0, int ld0, const void* g1, int ld1, const void* g2, int ld2,
                            const void* out, int out_ld, const void* y, int y_ld, int C, const double* stats,
                            const float* gamma, const float* beta, float eps, double* sums, float* dgamma, float* dbeta,
                            void* dy, int dy_ld, void* dres, int dres_ld, float* dbias, int N, int64_t nvox, void* stream) {
  SEG3D_REQUIRE(C > 0 && C % 8 == 0 && C <= GN_BWD_MAXC && 256 % (C / 8) == 0, "gn_bwd: unsupported C=%d", C);
  SEG3D_REQUIRE(g0 && y && stats && gamma && sums && N > 0 && nvox > 0, "gn_bwd: bad arguments");
  SEG3D_REQUIRE(out || beta, "gn_bwd: pass the saved output, or beta to recompute the ReLU mask from y (units without a residual)");
  SEG3D_REQUIRE(out || !dres, "gn_bwd: a unit with a residual needs its saved output for the ReLU mask");
  SEG3D_REQUIRE(pass == 0 ? (dgamma && dbeta) : (dy != nullptr), "gn_bwd: missing outputs for pass %d", pass);
  SEG3D_REQUIRE(ld0 % 8 == 0 && (!out || out_ld % 8 == 0) && y_ld % 8 == 0, "gn_bwd: pitches must be multiples of 8");
  const int cv = C / 8, vpb = 256 / cv;
  long long want = (nvox + vpb * 4 - 1) / (vpb * 4);
  const int sms = seg3d_num_sms();
  int gx = (int)(want < 1 ? 1 : (want > 4LL * sms ? 4LL * sms : want));
  dim3 grid(gx, N);
  cudaStream_t st = (cudaStream_t)stream;
#define SEG3D_GNB(PS, RM) gn_bwd_kernel<T, PS, RM><<<grid, 256, 0, st>>>((const T*)g0, ld0, (const T*)g1, ld1, (const T*)g2, ld2, (const T*)out, out_ld, \
        (const T*)y, y_ld, C, stats, gamma, beta, eps, sums, dgamma, dbeta, (T*)dy, dy_ld, (T*)dres, dres_ld, dbias, nvox)
  SEG3D_DISPATCH_DTYPE(dtype, T, {
    if (pass == 0) { if (out) SEG3D_GNB(0, false); else SEG3D_GNB(0, true); }
    else           { if (out) SEG3D_GNB(1, false); else SEG3D_GNB(1, true); }
  });
#undef SEG3D_GNB
  SEG3D_CHECK_LAUNCH("gn_bwd_kernel");
  return SEG3D_OK;
}

extern "C" int seg3d_gn_bwd_noact(int dtype, int pass, const void* g0, int ld0, const void* g1, int ld1, const void* g2, int ld2,
                                  const void* y, int y_ld, int C, const double* stats, const float* gamma, float eps,
                                  double* sums, float* dgamma, float* dbeta, void* dy, int dy_ld, void* dres, int dres_ld,
                                  float* dbias, int N, int64_t nvox, void* stream) {
  SEG3D_REQUIRE(C > 0 && C % 8 == 0 && C <= GN_BWD_MAXC && 256 % (C / 8) == 0, "gn_bwd_noact: unsupported C=%d", C);
  SEG3D_REQUIRE(g0 && y && stats && gamma && sums && N > 0 && nvox > 0, "gn_bwd_noact: bad arguments");
  SEG3D_REQUIRE(pass == 0 ? (dgamma && dbeta) : (dy != nullptr), "gn_bwd_noact: missing outputs for pass %d", pass);
  SEG3D_REQUIRE(ld0 % 8 == 0 && (!g1 || ld1 % 8 == 0) && (!g2 || ld2 % 8 == 0) && y_ld % 8 == 0,
                "gn_bwd_noact: pitches must be multiples of 8");
  SEG3D_REQUIRE(pass == 0 || (dy_ld % 8 == 0 && (!dres || dres_ld % 8 == 0)), "gn_bwd_noact: pitches must be multiples of 8");
  const int cv = C / 8, vpb = 256 / cv;
  long long want = (nvox + vpb * 4 - 1) / (vpb * 4);
  const int sms = seg3d_num_sms();
  int gx = (int)(want < 1 ? 1 : (want > 4LL * sms ? 4LL * sms : want));
  dim3 grid(gx, N);
  cudaStream_t st = (cudaStream_t)stream;
#define SEG3D_GNB(PS) gn_bwd_kernel<T, PS, false, true><<<grid, 256, 0, st>>>((const T*)g0, ld0, (const T*)g1, ld1, (const T*)g2, ld2, \
        (const T*)nullptr, 0, (const T*)y, y_ld, C, stats, gamma, nullptr, eps, sums, dgamma, dbeta, (T*)dy, dy_ld, (T*)dres, dres_ld, dbias, nvox)
  SEG3D_DISPATCH_DTYPE(dtype, T, {
    if (pass == 0) SEG3D_GNB(0); else SEG3D_GNB(1);
  });
#undef SEG3D_GNB
  SEG3D_CHECK_LAUNCH("gn_bwd_kernel");
  return SEG3D_OK;
}

int seg3d_wgrad_tc(int dtype, const void* x, int x_ld, int Cin, const void* dy, int dy_ld, int Cout, float* dw,
                   int N, int D, int H, int W, cudaStream_t st);
int seg3d_wgrad_tc9(int dtype, const void* x, int x_ld, int Cin, const void* dy, int dy_ld, int Cout, float* dw,
                    int N, int D, int H, int W, cudaStream_t st);
int seg3d_wgrad_s2_tc(int mode, int dtype, const void* x, int x_ld, int Cin, const void* dy, int dy_ld, int Cout, float* dw,
                      int N, int D, int H, int W, cudaStream_t st);

extern "C" int seg3d_conv3d_wgrad(int mode, int dtype, const void* x, int x_ld, int Cin, const void* dy, int dy_ld, int Cout,
                                  float* dw, int N, int D, int H, int W, void* stream) {
  SEG3D_REQUIRE(x && dy && dw && Cin > 0 && Cout > 0 && N > 0, "conv3d_wgrad: bad arguments");
  if (mode == SEG3D_CONV_K3 && Cin == 1 && Cout == 16 && x_ld == 1) {
    SEG3D_REQUIRE(dy_ld % 4 == 0 && ((uintptr_t)dy) % 16 == 0, "conv3d_wgrad(cin1): dy pitch / alignment");
    const int ntx = (W + 7) / 8, nty = (H + 7) / 8, ntz = (D + WC1_LZ - 1) / WC1_LZ;
    const long long ntiles = (long long)ntx * nty * ntz * N;
    const int gx = (int)(ntiles < (long long)seg3d_num_sms() ? ntiles : (long long)seg3d_num_sms());   // ~200 registers: one block per SM
    SEG3D_DISPATCH_DTYPE(dtype, T, (wgrad_cin1_kernel<T><<<gx, 256, 0, (cudaStream_t)stream>>>((const T*)x, (const T*)dy, dy_ld, dw, N, D, H, W, ntx, nty, ntz)));
    SEG3D_CHECK_LAUNCH("wgrad_cin1_kernel");
    return SEG3D_OK;
  }
  if (mode == SEG3D_CONV_K3) {       // tensor-core paths when the shape allows it: nine-taps-per-MMA for narrow outputs first
    const int rc9 = seg3d_wgrad_tc9(dtype, x, x_ld, Cin, dy, dy_ld, Cout, dw, N, D, H, W, (cudaStream_t)stream);
    if (rc9 != SEG3D_EUNSUPPORTED) return rc9;
    const int rc = seg3d_wgrad_tc(dtype, x, x_ld, Cin, dy, dy_ld, Cout, dw, N, D, H, W, (cudaStream_t)stream);
    if (rc != SEG3D_EUNSUPPORTED) return rc;
  }
  if (mode == SEG3D_CONV_K2S2 || mode == SEG3D_CONV_T2S2) {
    const int rc = seg3d_wgrad_s2_tc(mode, dtype, x, x_ld, Cin, dy, dy_ld, Cout, dw, N, D, H, W, (cudaStream_t)stream);
    if (rc != SEG3D_EUNSUPPORTED) return rc;
  }
  WgradGeom g;
  g.mode = mode; g.N = N; g.D = D; g.H = H; g.W = W; g.Cin = Cin; g.Cout = Cout; g.x_ld = x_ld; g.dy_ld = dy_ld;
  g.Do = D; g.Ho = H; g.Wo = W;
  int taps = 1;
  switch (mode) {
    case SEG3D_CONV_K3: taps = 27; break;
    case SEG3D_CONV_K1: taps = 1; break;
    case SEG3D_CONV_K2S2: taps = 8; g.Do = D / 2; g.Ho = H / 2; g.Wo = W / 2; break;
    case SEG3D_CONV_T2S2: taps = 8; break;
    default: seg3d_set_error("conv3d_wgrad: unknown mode %d", mode); return SEG3D_EINVAL;
  }
  const long long vps = (long long)g.Do * g.Ho * g.Wo;
  SEG3D_REQUIRE(vps > 0 && vps < (1ll << 31), "conv3d_wgrad: bad dims");
  g.vps = (int)vps;
  // voxels per CTA: aim at ~4 waves over the chip, at least 512 voxels per CTA to amortise the atomics
  const int tiles = ((Cin + 63) / 64) * ((Cout + 63) / 64);
  long long ctas_other = (long long)taps * tiles * N;
  long long want_chunks = (4LL * seg3d_num_sms() + ctas_other - 1) / ctas_other;
  if (want_chunks < 1) want_chunks = 1;
  long long chunk = (vps + want_chunks - 1) / want_chunks;
  if (chunk < 512) chunk = vps < 512 ? vps : 512;
  chunk = (chunk + 15) / 16 * 16;
  g.chunk = (int)chunk; g.nchunks = (int)((vps + chunk - 1) / chunk);
  dim3 grid((unsigned)(N * g.nchunks), taps, tiles);
  SEG3D_DISPATCH_DTYPE(dtype, T, (wgrad_simt_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>(g, (const T*)x, (const T*)dy, dw)));
  SEG3D_CHECK_LAUNCH("wgrad_simt_kernel");
  return SEG3D_OK;
}

extern "C" int seg3d_outblock_tail_bwd(int dtype, int pass, const void* y1, int ld, int C,
                                       const double* stats1, const float* gamma1, const float* beta1,
                                       const float* w2, const float* bias2,
                                       const double* stats2, const float* gamma2, const float* beta2, float eps,
                                       const float* dprobs, double* sums2, double* sums1,
                                       float* dgamma2, float* dbeta2, float* dw2, float* db2,
                                       float* dgamma1, float* dbeta1, float* db1,
                                       void* dy1, int dy_ld, int N, int64_t nvox, void* stream) {
  SEG3D_REQUIRE(y1 && stats1 && stats2 && gamma1 && beta1 && w2 && gamma2 && beta2 && dprobs && sums2 && sums1, "tail_bwd: bad arguments");
  SEG3D_REQUIRE(pass >= 0 && pass <= 2 && N > 0 && nvox > 0 && ld >= C, "tail_bwd: bad arguments");
  TailBwdArgs a;
  a.stats1 = stats1; a.stats2 = stats2; a.gamma1 = gamma1; a.beta1 = beta1; a.w2 = w2; a.bias2 = bias2; a.gamma2 = gamma2; a.beta2 = beta2;
  a.dprobs = dprobs; a.sums2 = sums2; a.sums1 = sums1; a.dgamma2 = dgamma2; a.dbeta2 = dbeta2; a.dw2 = dw2; a.db2 = db2;
  a.dgamma1 = dgamma1; a.dbeta1 = dbeta1; a.db1 = db1; a.eps = eps;
  const int sms = seg3d_num_sms();
  long long want = (nvox + 255) / 256;
  int gx = (int)(want < 1 ? 1 : (want > 2LL * sms ? 2LL * sms : want));
  dim3 grid(gx, N);
  cudaStream_t st = (cudaStream_t)stream;
  SEG3D_DISPATCH_DTYPE(dtype, T, {
    if (pass == 0) return launch_tail_bwd<T, 0>(C, grid, st, (const T*)y1, ld, a, (T*)dy1, dy_ld, nvox);
    if (pass == 1) return launch_tail_bwd<T, 1>(C, grid, st, (const T*)y1, ld, a, (T*)dy1, dy_ld, nvox);
    return launch_tail_bwd<T, 2>(C, grid, st, (const T*)y1, ld, a, (T*)dy1, dy_ld, nvox);
  });
  return SEG3D_OK;
}
