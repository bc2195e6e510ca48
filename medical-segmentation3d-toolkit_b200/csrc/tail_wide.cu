// tail_wide.cu - the output-block tail (GN1 + ReLU -> 1x1x1 conv (C x C) -> GN2 -> channel softmax) for 1 <= C <= 127
// classes on the tensor cores.  The SIMT tail (elementwise.cu) keeps a C-vector per thread and costs C^2 FMAs per voxel per
// pass; here the 1x1x1 conv of a 128-voxel tile is one 128 x Cp x Cp GEMM (Cp = 16 * ceil(C / 16)).
//
// Persistent, warp-specialised, one CTA per SM (its shared memory is sized so), each CTA owns a contiguous range of tiles:
//   warp 0      TMA: the raw out_block.conv1 rows of a tile (fp32, one sample, 128 voxels, channels in 32-wide boxes,
//               128B swizzle) into a stage of the ring; voxels past nvox and channels >= C arrive as zeros
//   warp 1      MMA: 3 * Cp / 16 MMAs of 128 x Cp x 16 per tile, hi*whi + lo*whi + hi*wlo into one fp32 TMEM accumulator
//   warps 2-5   transform: h = relu(fma(raw, a1, b1)) with GN1 folded per sample exactly as outblock_tail_kernel does,
//               split into hi = f16(h), lo = f16(h - hi), written IN PLACE over the stage as K-major 64B-swizzled UMMA rows
//               (box kb: hi rows in its first 8 KB, lo rows in its second 8 KB)
//   warps 6-17  epilogue: three groups of four warps, group g drains TMEM accumulator g (tiles g, g + 3, ...); one TMEM lane
//               is one voxel, so a thread owns a whole row and reads it in 16-column chunks.
//               pass 0: sum z and z^2 per sample (fp32 per thread, fp64 atomics once per warp per sample)
//               pass 1: three sweeps over the row - max, exp-sum, write - with the SIMT tail's expression sequence, stores
//               of 32 consecutive voxels per warp into probs[n][c][v]
// W2 is split into whi | wlo (f16) in shared memory once per CTA from the plan's fp32 [C][C] matrix.
#include "tc_ptx.cuh"

namespace {

constexpr int TW_THREADS = 576;
constexpr int TW_NG = 3;                 // epilogue groups = TMEM accumulators (a fourth group spills at 704 threads)
constexpr int TW_BOX = 16384;            // one 32-channel box of a tile: 128 rows x 128 B fp32 (= hi 8 KB + lo 8 KB after the transform)
constexpr int TW_MAXSTAGES = 8;

struct TwParams {
  int C, Cp, Kb, ns, tps, ntiles;        // classes, padded, 32-channel boxes, ring stages, tiles per sample, N * tps
  int nvox;
  float eps;
  uint32_t idesc, stage_bytes, b_off, tab_off, bar_off, tmem_cols, acc_pitch;   // acc_pitch: TMEM columns per accumulator
};

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

template <int PASS>
__global__ void __launch_bounds__(TW_THREADS, 1)
outblock_tail_wide_kernel(const __grid_constant__ CUtensorMap map_y, const TwParams p, const double* __restrict__ stats1,
                          const float* __restrict__ gamma1, const float* __restrict__ beta1, const float* __restrict__ w2,
                          const float* __restrict__ bias2, double* __restrict__ stats2, const float* __restrict__ gamma2,
                          const float* __restrict__ beta2, float* __restrict__ probs) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  float* sa1 = reinterpret_cast<float*>(smem_al + p.tab_off);            // [128] GN1 folded scale / shift (0 for c >= C)
  float* sb1 = sa1 + 128;
  float* sbias2 = sb1 + 128;                                              // [128]
  float* sa2 = sbias2 + 128;                                              // [TW_NG][128] GN2 folded, per epilogue group
  float* sb2 = sa2 + TW_NG * 128;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_al + p.bar_off);
  const uint32_t full_bar = smem_u32(bars);                               // [ns] TMA complete_tx
  const uint32_t afull_bar = full_bar + 8 * TW_MAXSTAGES;                 // [ns] 4 transform-warp arrivals
  const uint32_t empty_bar = afull_bar + 8 * TW_MAXSTAGES;                // [ns] tcgen05.commit
  const uint32_t tfull_bar = empty_bar + 8 * TW_MAXSTAGES;                // [TW_NG] tcgen05.commit
  const uint32_t tempty_bar = tfull_bar + 8 * TW_NG;                      // [TW_NG] 4 epilogue-warp arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * TW_MAXSTAGES + 2 * TW_NG);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.ns; ++s) { mbar_init(full_bar + 8 * s, 1); mbar_init(afull_bar + 8 * s, 4); mbar_init(empty_bar + 8 * s, 1); }
    for (int b = 0; b < TW_NG; ++b) { mbar_init(tfull_bar + 8 * b, 1); mbar_init(tempty_bar + 8 * b, 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x < 128) sbias2[threadIdx.x] = (bias2 && (int)threadIdx.x < p.C) ? bias2[threadIdx.x] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  // this CTA's tiles: [t0, t1), contiguous so a CTA meets few sample boundaries
  const int t0 = (int)(((long long)p.ntiles * blockIdx.x) / gridDim.x);
  const int t1 = (int)(((long long)p.ntiles * (blockIdx.x + 1)) / gridDim.x);
  const int ksteps = p.Cp >> 4;

  if (warp == 0) {
    // ===== TMA producer =====
    int n = t0 / p.tps, i = t0 - n * p.tps;
    int stage = 0; uint32_t phase = 0;
    for (int t = t0; t < t1; ++t) {
      mbar_wait(empty_bar + 8 * stage, phase ^ 1);
      const uint32_t dst = smem_base + (uint32_t)stage * p.stage_bytes;
      mbar_expect_tx_e(full_bar + 8 * stage, (uint32_t)p.Kb * TW_BOX);
      for (int kb = 0; kb < p.Kb; ++kb)
        if (elect_one()) tma_load_3d(dst + kb * TW_BOX, &map_y, full_bar + 8 * stage, kb * 32, i * 128, n);
      if (++stage == p.ns) { stage = 0; phase ^= 1; }
      if (++i == p.tps) { i = 0; ++n; }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (whole warp, converged: see elect_one()) =====
    const uint32_t hi = desc_hi(512, 4);                  // 8-row groups 512 B apart, 64B swizzle
    const uint32_t b_hi = (smem_base + p.b_off) >> 4, b_lo_step = (uint32_t)(p.Kb * p.Cp * 64) >> 4;
    const uint32_t b_kstep = (uint32_t)(p.Cp * 64) >> 4;
    int stage = 0; uint32_t phase = 0;
    int buf = 0; uint32_t bphase = 0;
    for (int t = t0; t < t1; ++t) {
      mbar_wait(tempty_bar + 8 * buf, bphase ^ 1);
      mbar_wait(afull_bar + 8 * stage, phase);
      tc_fence_after();
      const uint32_t a0 = (smem_base + (uint32_t)stage * p.stage_bytes) >> 4;
      const uint32_t d = tmem_base + (uint32_t)buf * p.acc_pitch;
      for (int ks = 0; ks < ksteps; ++ks) {
        const uint32_t kb = (uint32_t)ks >> 1, off = ((uint32_t)ks & 1u) * 2u;      // 32 B = 16 K-values into the 64 B row
        const uint32_t ahi = a0 + kb * (TW_BOX >> 4) + off, alo = ahi + (8192 >> 4);
        const uint32_t bhi = b_hi + kb * b_kstep + off, blo = bhi + b_lo_step;
        tc_mma_f16_e(d, desc_pack(hi, ahi), desc_pack(hi, bhi), p.idesc, ks > 0 ? 1u : 0u);
        tc_mma_f16_e(d, desc_pack(hi, alo), desc_pack(hi, bhi), p.idesc, 1u);
        tc_mma_f16_e(d, desc_pack(hi, ahi), desc_pack(hi, blo), p.idesc, 1u);
      }
      tc_commit_e(empty_bar + 8 * stage);
      tc_commit_e(tfull_bar + 8 * buf);
      if (++stage == p.ns) { stage = 0; phase ^= 1; }
      if (++buf == TW_NG) { buf = 0; bphase ^= 1; }
    }
  } else if (warp <= 5) {
    // ===== transform =====
    const int r = (warp - 2) * 32 + lane;                 // tile row = voxel
    // B = [whi | wlo] rows o (output class), K = input class, 64B-swizzled blocks of 32 K-values: [hl][kb][Cp rows][64 B]
    {
      const int nchunk = p.Kb * p.Cp * 4;
      uint8_t* bbase = smem_al + p.b_off;
      for (int q = r; q < nchunk; q += 128) {
        const int c = q & 3, o = (q >> 2) % p.Cp, kb = (q >> 2) / p.Cp;
        float wv[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int k = kb * 32 + c * 8 + e;
          wv[e] = (o < p.C && k < p.C) ? w2[o * p.C + k] : 0.f;
        }
        uint32_t hw[4], lw[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const __half h0 = __float2half_rn(wv[2 * e]), h1 = __float2half_rn(wv[2 * e + 1]);
          hw[e] = pack_h2(__half2float(h0), __half2float(h1));
          lw[e] = pack_h2(wv[2 * e] - __half2float(h0), wv[2 * e + 1] - __half2float(h1));
        }
        const int boff = (kb * p.Cp + o) * 64 + ((c ^ ((o >> 1) & 3)) << 4);
        *reinterpret_cast<uint4*>(bbase + boff) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
        *reinterpret_cast<uint4*>(bbase + p.Kb * p.Cp * 64 + boff) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
      }
    }
    int n = t0 / p.tps, i = t0 - n * p.tps, cur_n = -1;
    int stage = 0; uint32_t phase = 0;
    const int sw_in = r & 7, sw_out = (r >> 1) & 3;
    for (int t = t0; t < t1; ++t) {
      if (n != cur_n) {                                   // fold GN1 of sample n (outblock_tail_kernel's expression)
        named_bar_sync(1, 128);
        {
          float mean, rstd;
          gn_mean_rstd(stats1 + 2 * n, (double)p.nvox * p.C, p.eps, mean, rstd);
          const float a = r < p.C ? rstd * gamma1[r] : 0.f;
          sa1[r] = a; sb1[r] = r < p.C ? beta1[r] - mean * a : 0.f;
        }
        named_bar_sync(1, 128);
        cur_n = n;
      }
      mbar_wait_relaxed(full_bar + 8 * stage, phase);
      uint8_t* sbase = smem_al + (size_t)stage * p.stage_bytes;
      for (int kb = 0; kb < p.Kb; ++kb) {
        uint8_t* box = sbase + kb * TW_BOX;
        float v[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 f = *reinterpret_cast<const float4*>(box + r * 128 + ((j ^ sw_in) << 4));
          v[4 * j] = f.x; v[4 * j + 1] = f.y; v[4 * j + 2] = f.z; v[4 * j + 3] = f.w;
        }
        named_bar_sync(1, 128);                           // every row of the box is read before the hi / lo rows overwrite it
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t hw[4], lw[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int ch = kb * 32 + c * 8 + 2 * e;
            const float h0 = fmaxf(fmaf(v[c * 8 + 2 * e], sa1[ch], sb1[ch]), 0.f);
            const float h1 = fmaxf(fmaf(v[c * 8 + 2 * e + 1], sa1[ch + 1], sb1[ch + 1]), 0.f);
            const float q0 = __half2float(__float2half_rn(h0)), q1 = __half2float(__float2half_rn(h1));
            hw[e] = pack_h2(q0, q1);
            lw[e] = pack_h2(h0 - q0, h1 - q1);
          }
          const int o = r * 64 + ((c ^ sw_out) << 4);
          *reinterpret_cast<uint4*>(box + o) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          *reinterpret_cast<uint4*>(box + 8192 + o) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(afull_bar + 8 * stage);
      if (++stage == p.ns) { stage = 0; phase ^= 1; }
      if (++i == p.tps) { i = 0; ++n; }
    }
  } else {
    // ===== epilogue =====
    const int g = (warp - 6) >> 2, q = warp & 3;          // group g owns TMEM accumulator g; q = the warp's TMEM lane quarter
    const int r = q * 32 + lane;
    float* ga2 = sa2 + g * 128;
    float* gb2 = sb2 + g * 128;
    const int C = p.C;
    int t = t0 + g;
    int n = t / p.tps, i = t - n * p.tps, cur_n = -1;
    uint32_t ph = 0;
    float s = 0.f, ss = 0.f;
    const uint32_t tcol0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)g * p.acc_pitch;
    for (; t < t1; t += TW_NG) {
      if (n != cur_n) {
        if (PASS == 0) {
          if (cur_n >= 0) {
            s = warp_sum(s); ss = warp_sum(ss);
            if (lane == 0) { atomicAdd(stats2 + 2 * cur_n, (double)s); atomicAdd(stats2 + 2 * cur_n + 1, (double)ss); }
            s = 0.f; ss = 0.f;
          }
        } else {
          named_bar_sync(2 + g, 128);
          float mean, rstd;
          gn_mean_rstd(stats2 + 2 * n, (double)p.nvox * C, p.eps, mean, rstd);
          const float a = r < C ? rstd * gamma2[r] : 0.f;
          ga2[r] = a; gb2[r] = r < C ? beta2[r] - mean * a : 0.f;
          named_bar_sync(2 + g, 128);
        }
        cur_n = n;
      }
      mbar_wait_relaxed(tfull_bar + 8 * g, ph);
      tc_fence_after();
      const int v = i * 128 + r;
      const bool valid = v < p.nvox;
      uint32_t x[16];
      if (PASS == 0) {
        for (int cc = 0; cc < ksteps; ++cc) {
          tc_ld16(tcol0 + (uint32_t)(cc * 16), x);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int c = cc * 16 + j;
            if (valid && c < C) {
              const float z = __uint_as_float(x[j]) + sbias2[c];
              s += z; ss += z * z;
            }
          }
        }
      } else {
        float m = -INFINITY;
        for (int cc = 0; cc < ksteps; ++cc) {
          tc_ld16(tcol0 + (uint32_t)(cc * 16), x);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int c = cc * 16 + j;
            if (c < C) m = fmaxf(m, fmaf(__uint_as_float(x[j]) + sbias2[c], ga2[c], gb2[c]));
          }
        }
        float den = 0.f;
        for (int cc = 0; cc < ksteps; ++cc) {
          tc_ld16(tcol0 + (uint32_t)(cc * 16), x);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int c = cc * 16 + j;
            if (c < C) den += expf(fmaf(__uint_as_float(x[j]) + sbias2[c], ga2[c], gb2[c]) - m);
          }
        }
        const float inv = 1.f / den;
        float* dst = probs + (size_t)n * C * p.nvox + v;
        for (int cc = 0; cc < ksteps; ++cc) {
          tc_ld16(tcol0 + (uint32_t)(cc * 16), x);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int c = cc * 16 + j;
            if (valid && c < C) dst[(size_t)c * p.nvox] = expf(fmaf(__uint_as_float(x[j]) + sbias2[c], ga2[c], gb2[c]) - m) * inv;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar + 8 * g);
      ph ^= 1;
      i += TW_NG;
      while (i >= p.tps) { i -= p.tps; ++n; }
    }
    if (PASS == 0 && cur_n >= 0) {
      s = warp_sum(s); ss = warp_sum(ss);
      if (lane == 0) { atomicAdd(stats2 + 2 * cur_n, (double)s); atomicAdd(stats2 + 2 * cur_n + 1, (double)ss); }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

}  // namespace

extern "C" int seg3d_outblock_tail_wide(int pass, const float* y1, int ld, int C, const double* stats1, const float* gamma1,
                                        const float* beta1, const float* w2, const float* bias2, float eps, double* stats2,
                                        const float* gamma2, const float* beta2, float* probs, int N, int64_t nvox, void* stream) {
  if (C < 1 || C > 127) { seg3d_set_error("outblock_tail_wide: C=%d not in 1..127 (the int8 label mask holds 127 classes)", C); return SEG3D_EUNSUPPORTED; }
  if (((uintptr_t)y1) % 16 != 0 || ld % 4 != 0) {
    seg3d_set_error("outblock_tail_wide: y1 must be 16-byte aligned with a pitch that is a multiple of 4 floats (ld=%d)", ld);
    return SEG3D_EUNSUPPORTED;
  }
  SEG3D_REQUIRE(pass == 0 || pass == 1, "outblock_tail_wide: pass must be 0 (GN2 sums) or 1 (probabilities)");
  SEG3D_REQUIRE(y1 && stats1 && gamma1 && beta1 && w2 && stats2 && N > 0 && nvox > 0 && ld >= C, "outblock_tail_wide: bad arguments");
  SEG3D_REQUIRE(pass == 0 || (gamma2 && beta2 && probs), "outblock_tail_wide: pass 1 needs gamma2, beta2 and probs");
  SEG3D_REQUIRE(nvox < (1ll << 31) - 128, "outblock_tail_wide: nvox=%lld out of range", (long long)nvox);
  EncodeTiledFn encode = get_encode();
  if (!encode) { seg3d_set_error("outblock_tail_wide: cuTensorMapEncodeTiled entry point not available"); return SEG3D_ECUDA; }

  TwParams p;
  memset(&p, 0, sizeof(p));
  p.C = C; p.Cp = (C + 15) & ~15; p.Kb = (p.Cp + 31) / 32;
  p.nvox = (int)nvox; p.eps = eps;
  p.tps = (int)((nvox + 127) / 128);
  const long long ntiles = (long long)N * p.tps;
  SEG3D_REQUIRE(ntiles < (1ll << 31), "outblock_tail_wide: tile count out of range");
  p.ntiles = (int)ntiles;
  p.stage_bytes = (uint32_t)p.Kb * TW_BOX;
  const uint32_t b_bytes = 2u * p.Kb * p.Cp * 64;
  // ring stages: fill ~200 KB, which also keeps the kernel at one CTA per SM (its TMEM allocation assumes that)
  int ns = (int)((200 * 1024 - b_bytes) / p.stage_bytes);
  if (ns > TW_MAXSTAGES) ns = TW_MAXSTAGES;
  p.ns = ns;
  p.b_off = (uint32_t)ns * p.stage_bytes;
  p.tab_off = p.b_off + b_bytes;
  p.bar_off = p.tab_off + (3 + 2 * TW_NG) * 128 * 4;
  const size_t smem = 1024 + (size_t)p.bar_off + (3 * TW_MAXSTAGES + 2 * TW_NG) * 8 + 16;
  SEG3D_REQUIRE(ns >= 2 && smem > 116 * 1024, "outblock_tail_wide: shared-memory plan failed (C=%d)", C);
  p.acc_pitch = 16;
  while (p.acc_pitch < (uint32_t)p.Cp) p.acc_pitch <<= 1;
  p.tmem_cols = 32;                                       // tcgen05.alloc takes a power of two >= 32
  while (p.tmem_cols < TW_NG * p.acc_pitch) p.tmem_cols <<= 1;
  p.idesc = (1u << 4) | ((uint32_t)(p.Cp >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);    // f16 x f16 -> f32, K-major A and B

  CUtensorMap map;
  cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)nvox, (cuuint64_t)N};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)nvox * ld * 4};
  cuuint32_t box[3] = {32, 128, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = encode(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(y1), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { seg3d_set_error("outblock_tail_wide: cuTensorMapEncodeTiled failed with %d", (int)r); return SEG3D_ECUDA; }

  const int sms = seg3d_num_sms();
  dim3 grid((unsigned)(p.ntiles < sms ? p.ntiles : sms));
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e;
  if (pass == 0) {
    e = cudaFuncSetAttribute(outblock_tail_wide_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess)
      outblock_tail_wide_kernel<0><<<grid, TW_THREADS, smem, st>>>(map, p, stats1, gamma1, beta1, w2, bias2, stats2, nullptr, nullptr, nullptr);
  } else {
    e = cudaFuncSetAttribute(outblock_tail_wide_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess)
      outblock_tail_wide_kernel<1><<<grid, TW_THREADS, smem, st>>>(map, p, stats1, gamma1, beta1, w2, bias2, stats2, gamma2, beta2, probs);
  }
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { seg3d_set_error("outblock_tail_wide_kernel launch failed: %s", cudaGetErrorString(e)); return SEG3D_ECUDA; }
  return SEG3D_OK;
}
