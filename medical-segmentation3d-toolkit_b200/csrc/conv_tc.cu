// conv_tc.cu - k=3 s=1 p=1 Conv3d as an implicit GEMM on the 5th-gen tensor cores (sm_100a).
//
//   D[128 voxels x Cout] (fp32, TMEM)  +=  A[128 voxels x KC] (smem, K-major)  *  B[Cout x KC]^T (smem, K-major)
//
// summed over the 27 filter taps and the Cin/KC channel chunks.  One CTA owns one output tile: a
// tw x th x td box of voxels (tw*th*td = 128) of one sample.  For every (tap, chunk) the TMA
// producer warp loads the box shifted by the tap offset from the NDHWC activation tensor through
// a 5-D tensor map - out-of-bounds coordinates are zero-filled by the TMA unit, which IS the
// "same" padding - and the matching [Cout x KC] weight slab through a 2-D map.  Both land in
// 128B/64B/32B-swizzled K-major layouts that tcgen05.mma consumes through shared-memory
// descriptors.  One elected thread issues the MMAs; the accumulator lives in TMEM; four epilogue
// warps read it back with tcgen05.ld, add the bias, take the GroupNorm partial sums from the
// fp32 values, and store fp16/bf16 NDHWC rows with 16-byte stores.
//
// Warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2.. = epilogue (TMEM lane quarter =
// warp_id % 4; the forward kernels run 8 epilogue warps, two per quarter, splitting the accumulator columns).
// Kernels in this file: conv3d_tc_persistent_kernel (generic k3 / k2s2 / transposed, persistent, double-buffered
// TMEM), conv3d_k3_zmarch_kernel (narrow k3 layers, resident weights, halo-plane reuse), conv3d_k3_wgrad_tc_kernel and
// conv3d_s2_wgrad_tc_kernel (weight gradients, MN-major operands).
#include "tc_ptx.cuh"

namespace {

constexpr int g_kwfuse_default = 1;
constexpr int TCE_THREADS = 320;     // forward kernels: TMA warp, MMA warp, 8 epilogue warps (two per TMEM lane quarter)

struct TcParams {
  int Cin, Cout, KC, nchunk;        // KC = channels per K block, nchunk = Cin / KC
  int D, H, W, N;
  int tw, th, td;                   // tile box
  int ntx, nty, ntz;                // tiles per axis
  int y_ld;
  int stages, a_bytes, b_bytes;     // per-stage operand slab pitches (1024-aligned)
  int tx_bytes;                     // bytes the two TMA loads of one stage actually write
  int tmem_cols;
  uint32_t idesc;
  uint32_t sbo;                     // B operand: stride between 8-row groups, bytes
  uint32_t a_sbo;                   // A operand: stride between 8-row groups (one x-line of the box), bytes
  uint32_t layout_type;             // UMMA smem descriptor swizzle code
  int kwfuse;                       // 1: one A box (tw+2 wide) per (kd,kh) serves the three kw taps via x-shifted descriptors
  int b_slab;                       // pitch of one kw weight slab inside a stage (kwfuse)
  int row_bytes;
  int conv;                         // 0: k3 s1 p1, 1: k2 s2 (folded-stride tensor map), 2: transposed k2 s2
  int cout_real, npass;             // transposed conv: real Cout; GEMM N = 8*Cout split into npass passes of p.Cout columns
  int ntaps;                        // outer tap count of the K loop (27, 9 when kw-fused, 8 for k2s2)
  int x_ld, halfW, halfH;           // k2s2 coordinate folding
  int ntiles, acc_cols;             // persistent kernel: total tiles, TMEM columns per accumulator buffer
  int wide;                         // epilogue may use 256-bit stores (32-byte aligned rows)
  // GroupNorm folded into the epilogue of a conv that is cheap to run twice (HBM-bound stride-2 / transposed convs):
  // epi_mode 0: store raw + statistics; 1: statistics only, nothing stored; 2: y = relu(gn(conv)) from finished statistics
  // split-operand strict mode: activations are [hi | lo] f16 halves (lo_off channels apart), weights [whi | wlo]; the K loop runs
  // the three products hi*whi, lo*whi, hi*wlo, so the fp32 accumulator carries ~22-bit operands
  int split, lo_off, nchunk_real;
  int out_f32;                      // store the fp32 accumulator (+bias) as float rows of pitch y_ld instead of T
  int epi_mode;
  float gn_eps;
  double gn_count;                  // elements per sample of the GroupNorm(1,C) input = real Cout * output voxels
  const double* gn_stats;           // [N][2] finished sums (epi_mode 2)
  const float* gn_gamma;
  const float* gn_beta;
};

// Persistent variant: each CTA walks tiles blockIdx.x, +gridDim.x, ...; the operand ring keeps
// streaming across tile boundaries and two TMEM accumulator buffers let the epilogue of tile i
// overlap the MMAs of tile i+1.  GroupNorm partial sums stay in registers until the sample changes.
template <typename T, int KC>
__global__ void __launch_bounds__(TCE_THREADS)
conv3d_tc_persistent_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                            const TcParams p, const float* __restrict__ bias, T* __restrict__ y, double* __restrict__ stats) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t a_base = smem_base;
  const uint32_t b_base = smem_base + p.stages * p.a_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_al + p.stages * (p.a_bytes + p.b_bytes));
  const uint32_t full_bar = smem_u32(bars);                   // [stages]
  const uint32_t empty_bar = full_bar + 8 * p.stages;         // [stages]
  const uint32_t tfull_bar = empty_bar + 8 * p.stages;        // [2]
  const uint32_t tempty_bar = tfull_bar + 16;                 // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * p.stages + 4);
  float* sbias = reinterpret_cast<float*>(tmem_slot + 4);     // [cout_real] bias (zeros when there is none), 16-byte aligned

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler
  for (int c = threadIdx.x; c < p.cout_real; c += blockDim.x) sbias[c] = bias ? bias[c] : 0.f;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    for (int s = 0; s < p.stages; ++s) { mbar_init(full_bar + 8 * s, 1); mbar_init(empty_bar + 8 * s, 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar + 8 * b, 1); mbar_init(tempty_bar + 8 * b, 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  const int kiters = p.ntaps * p.nchunk;

  if (warp == 0) {
    {   // whole warp, converged: see elect_one()
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        int t = tile;
        const int pass = t % p.npass; t /= p.npass;
        const int x0 = (t % p.ntx) * p.tw; t /= p.ntx;
        const int y0 = (t % p.nty) * p.th; t /= p.nty;
        const int z0 = (t % p.ntz) * p.td; const int n = t / p.ntz;
        for (int it = 0; it < kiters; ++it) {
          const int tap = it / p.nchunk, ck = it - tap * p.nchunk;
          int a_c = ck * p.KC, w_c = ck * p.KC;                 // channel coordinates of this K chunk in x and in w
          if (p.split) {
            const int ps = ck / p.nchunk_real, c = ck - ps * p.nchunk_real;
            a_c = c * p.KC + (ps == 1 ? p.lo_off : 0);
            w_c = c * p.KC + (ps == 2 ? p.Cin : 0);
          }
          mbar_wait(empty_bar + 8 * stage, phase ^ 1);
          mbar_expect_tx_e(full_bar + 8 * stage, (uint32_t)p.tx_bytes);
          const uint32_t fb = full_bar + 8 * stage, sa = a_base + stage * p.a_bytes, sb = b_base + stage * p.b_bytes;
          if (p.conv == 2) {         // transposed conv: plain GEMM rows, weight rows of this N-pass
            tma_load_5d_e(sa, &map_x, fb, a_c, x0, y0, z0, n);
            tma_load_2d_e(sb, &map_w, fb, w_c, pass * p.Cout);
          } else if (p.conv == 1) {  // k2 s2: tap = (kd*2+kh)*2+kw folded into the (channel, x, y) coordinates
            const int kd = tap >> 2, kh = (tap >> 1) & 1, kw = tap & 1;
            tma_load_5d_e(sa, &map_x, fb, kw * p.x_ld + a_c, x0 + kh * p.halfW, y0 + kd * p.halfH, z0, n);
            tma_load_2d_e(sb, &map_w, fb, w_c, tap * p.Cout);
          } else if (p.kwfuse) {
            const int kd = tap / 3, kh = tap % 3;
            tma_load_5d_e(sa, &map_x, fb, a_c, x0 - 1, y0 + kh - 1, z0 + kd - 1, n);
            for (int kw = 0; kw < 3; ++kw)
              tma_load_2d_e(sb + kw * p.b_slab, &map_w, fb, w_c, (tap * 3 + kw) * p.Cout);
          } else {
            const int kd = tap / 9, kh = (tap / 3) % 3, kw = tap % 3;
            tma_load_5d_e(sa, &map_x, fb, a_c, x0 + kw - 1, y0 + kh - 1, z0 + kd - 1, n);
            tma_load_2d_e(sb, &map_w, fb, w_c, tap * p.Cout);
          }
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {   // whole warp, converged: see elect_one()
      int stage = 0; uint32_t phase = 0; int j = 0;
      constexpr int KSTEPS = KC / 16;
      constexpr uint32_t ROWB = KC * 2;
      const bool fused = (p.conv == 0 && p.kwfuse);
      const uint32_t hi_a = desc_hi(p.a_sbo, p.layout_type), hi_b = desc_hi(p.sbo, p.layout_type);
      const uint32_t slab16 = (uint32_t)p.b_slab >> 4;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++j) {
        const int buf = j & 1;
        mbar_wait(tempty_bar + 8 * buf, ((j >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t dcol = tmem_base + (uint32_t)(buf * p.acc_cols);
        for (int it = 0; it < kiters; ++it) {
          mbar_wait(full_bar + 8 * stage, phase);
          tc_fence_after();
          const uint32_t lo_a = (a_base + stage * p.a_bytes) >> 4, lo_b = (b_base + stage * p.b_bytes) >> 4;
          if (fused) {
#pragma unroll
            for (int kw = 0; kw < 3; ++kw)
#pragma unroll
              for (int k = 0; k < KSTEPS; ++k)
                tc_mma_f16_e(dcol, desc_pack(hi_a, lo_a + ((kw * ROWB + k * 32) >> 4)), desc_pack(hi_b, lo_b + kw * slab16 + ((k * 32) >> 4)),
                           p.idesc, (it | kw | k) != 0);
          } else {
#pragma unroll
            for (int k = 0; k < KSTEPS; ++k)
              tc_mma_f16_e(dcol, desc_pack(hi_a, lo_a + ((k * 32) >> 4)), desc_pack(hi_b, lo_b + ((k * 32) >> 4)), p.idesc, (it | k) != 0);
          }
          tc_commit_e(empty_bar + 8 * stage);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
        tc_commit_e(tfull_bar + 8 * buf);
      }
    }
  } else {
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;             // warps 2-5 take the even 16-column chunks, warps 6-9 the odd ones
    const int r = q * 32 + lane;
    const int lx = r % p.tw, ly = (r / p.tw) % p.th, lz = r / (p.tw * p.th);
    float s = 0.f, ss = 0.f;
    int cur_n = -1, j = 0, gn_n = -1;
    float gn_mean = 0.f, gn_rstd = 1.f;
    const bool wide = p.wide != 0;
    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++j) {
      int t = tile;
      const int pass = t % p.npass; t /= p.npass;
      const int x0 = (t % p.ntx) * p.tw; t /= p.ntx;
      const int y0 = (t % p.nty) * p.th; t /= p.nty;
      const int z0 = (t % p.ntz) * p.td; const int n = t / p.ntz;
      if (stats && n != cur_n) {
        if (cur_n >= 0) {
          s = warp_sum(s); ss = warp_sum(ss);
          if (lane == 0) { atomicAdd(stats + 2 * cur_n, (double)s); atomicAdd(stats + 2 * cur_n + 1, (double)ss); }
        }
        s = 0.f; ss = 0.f; cur_n = n;
      }
      if (p.epi_mode == 2 && n != gn_n) { gn_mean_rstd(p.gn_stats + 2 * n, p.gn_count, p.gn_eps, gn_mean, gn_rstd); gn_n = n; }
      const int gx = x0 + lx, gy = y0 + ly, gz = z0 + lz;
      const bool valid = (gx < p.W) && (gy < p.H) && (gz < p.D);      // W/H/D = OUTPUT dims here
      const size_t vox = (((size_t)n * p.D + gz) * p.H + gy) * p.W + gx;
      T* yrow = y + vox * p.y_ld;
      const int buf = j & 1;
      mbar_wait(tfull_bar + 8 * buf, (j >> 1) & 1);
      tc_fence_after();
      const uint32_t tcol = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * p.acc_cols);
      // this warp's 16-column chunks: half, half+2, ...; the TMEM load of the next chunk is in flight while the
      // current one is converted and stored
      // t2s2: column -> (tap, co), output voxel (2z+kd, 2y+kh, 2x+kw): one 64-bit base per tile, 32-bit tap offsets per chunk
      T* ybase = yrow;
      if (p.conv == 2) {
        const size_t ov0 = (((size_t)n * 2 * p.D + 2 * gz) * 2 * p.H + 2 * gy) * 2 * p.W + 2 * gx;
        ybase = y + ov0 * p.y_ld;
      }
      if (p.out_f32)      // the output is a float tensor: redo the row base in float elements (T is 2 bytes wide)
        ybase = reinterpret_cast<T*>(reinterpret_cast<float*>(y) + (ybase - y));
      auto emit = [&](const uint32_t* v, int c0) {
        float f[16];
        int co = c0, off = c0;
        if (p.conv == 2) {
          const int col = pass * p.Cout + c0;
          const int tap = col / p.cout_real; co = col - tap * p.cout_real;
          off = (((tap >> 2) * 2 * p.H + ((tap >> 1) & 1)) * 2 * p.W + (tap & 1)) * p.y_ld + co;
        }
        const float4* b4 = reinterpret_cast<const float4*>(sbias + co);
#pragma unroll
        for (int jj = 0; jj < 16; jj += 4) {
          const float4 bb = b4[jj >> 2];
          f[jj] = __uint_as_float(v[jj]) + bb.x; f[jj + 1] = __uint_as_float(v[jj + 1]) + bb.y;
          f[jj + 2] = __uint_as_float(v[jj + 2]) + bb.z; f[jj + 3] = __uint_as_float(v[jj + 3]) + bb.w;
        }
        if (valid) {
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) { s += f[jj]; ss = fmaf(f[jj], f[jj], ss); }
        }
        if (p.epi_mode == 2) {
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) {
            const float a = gn_rstd * p.gn_gamma[co + jj];
            f[jj] = fmaxf(fmaf(f[jj], a, p.gn_beta[co + jj] - gn_mean * a), 0.f);
          }
        }
        if (valid && p.epi_mode != 1) {
          if (p.out_f32) {
            float4* d4 = reinterpret_cast<float4*>(reinterpret_cast<float*>(ybase) + off);     // ybase / off in elements of the fp32 tensor
#pragma unroll
            for (int jj = 0; jj < 16; jj += 4) d4[jj >> 2] = make_float4(f[jj], f[jj + 1], f[jj + 2], f[jj + 3]);
          } else {
            store16<T>(ybase + off, f, wide);
          }
        }
      };
      uint32_t va[16], vb[16];
      int c0 = half * 16;
      if (c0 < p.Cout) tc_ld16(tcol + (uint32_t)c0, va);
      while (c0 < p.Cout) {
        tc_wait_ld();
        if (c0 + 32 < p.Cout) tc_ld16(tcol + (uint32_t)(c0 + 32), vb);
        emit(va, c0);
        c0 += 32;
        if (c0 >= p.Cout) break;
        tc_wait_ld();
        if (c0 + 32 < p.Cout) tc_ld16(tcol + (uint32_t)(c0 + 32), va);
        emit(vb, c0);
        c0 += 32;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar + 8 * buf);
    }
    if (stats && cur_n >= 0) {
      s = warp_sum(s); ss = warp_sum(ss);
      if (lane == 0) { atomicAdd(stats + 2 * cur_n, (double)s); atomicAdd(stats + 2 * cur_n + 1, (double)ss); }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}


// ---------------------------------------------------------------------------------------------------
// z-marching variant for the narrow layers (Cin <= 64 in one K block, all 27 weight slabs resident in
// shared memory).  A CTA owns an 8(x) x 16(y) column and walks along z: every input plane (a
// 10 x 18 voxel halo box, one TMA load) is read from L2 exactly once and feeds the three output planes
// z-1, z, z+1 through 27 row-shifted descriptors (the 128B/64B/32B swizzle is a function of the absolute
// shared-memory address, so any row-aligned start address addresses the halo correctly).  nb TMEM
// accumulators rotate: three receive MMAs while the others are drained by the epilogue warps.
// L2->SM traffic per output voxel drops from 27 (per-tap boxes) to ~1.5 voxel reads.
// At M=128 an MMA re-reads its 128 x 16 A rows from shared memory (32 cycles) whatever N is, so N <= 32 is
// A-feed bound at half the tensor rate.  The three output planes an input plane contributes to sit in adjacent
// accumulators and the weight slabs are stored [(kh,kw)][kd=2,1,0][Cout][Cin], so ONE MMA with N = 3*Cout covers
// all three kd taps of a (kh,kw) position: 9*Cin/16 MMAs per plane instead of 27*Cin/16, each math-bound.
struct ZmParams {
  int Cout, KC, row_bytes;
  int D, H, W, N, y_ld;
  int ntx, nty, nseg, lseg, nitems;
  int ring, plane_bytes, w_slab, plane_tx, w_tx;
  int acc_cols, tmem_cols;
  int nb, maxblk;                   // rotating TMEM accumulators; output planes one MMA may cover (N = maxblk * Cout)
  int wide;                         // epilogue may use 256-bit stores
  int out_f32;                      // store the raw conv result as fp32 (out_block.conv1: its rounding would dominate the probability error)
  uint32_t idesc0, n8, sbo, a_sbo, layout_type;   // instruction descriptor without N; N/8 of one block (Cout >> 3)
  // XF: the first xf_nch input channels are a RAW convolution result whose GroupNorm(1, xf_nch) + ReLU has not been applied:
  // four transform warps form relu(gn(raw)) in place in every loaded halo plane (finished sums xf_stats, per sample)
  int xf_nch;
  float xf_eps;
  double xf_count;
  const double* xf_stats;
  const float* xf_gamma;
  const float* xf_beta;
};
constexpr int ZM_MAXNB = 8;
constexpr int ZMX_THREADS = TCE_THREADS + 128;

// SPLIT (strict-parity mode, seg3d_conv3d_split_fwd): the KC channels of a voxel row are [hi(KC/2) | lo(KC/2)] f16 halves of the
// activation, a weight row is [whi(KC/2) | wlo(KC/2)], and the k loop runs the three products hi*whi, lo*whi, hi*wlo
// (A k-step, B k-step) instead of the diagonal - the plane, the slabs and the N-fold over three output planes are unchanged.
template <typename T, int KC, bool SPLIT, bool XF = false>
__global__ void __launch_bounds__(XF ? ZMX_THREADS : TCE_THREADS)
conv3d_k3_zmarch_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                        const ZmParams p, const float* __restrict__ bias, T* __restrict__ y, double* __restrict__ stats) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t w_base = smem_base;
  const uint32_t a_base = smem_base + 27 * p.w_slab;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_al + 27 * p.w_slab + p.ring * p.plane_bytes);
  const uint32_t full_bar = smem_u32(bars);                   // [ring]
  const uint32_t empty_bar = full_bar + 8 * p.ring;           // [ring]
  const uint32_t tfull_bar = empty_bar + 8 * p.ring;          // [ZM_MAXNB]
  const uint32_t tempty_bar = tfull_bar + 8 * ZM_MAXNB;       // [ZM_MAXNB]
  const uint32_t wfull_bar = tempty_bar + 8 * ZM_MAXNB;       // [1]
  const uint32_t xf_bar = wfull_bar + 8;                      // [ring] plane transformed (XF)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * p.ring + 2 * ZM_MAXNB + 1);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    for (int s = 0; s < p.ring; ++s) { mbar_init(full_bar + 8 * s, 1); mbar_init(empty_bar + 8 * s, 1); mbar_init(xf_bar + 8 * s, 4); }
    for (int b = 0; b < ZM_MAXNB; ++b) { mbar_init(tfull_bar + 8 * b, 1); mbar_init(tempty_bar + 8 * b, 8); }
    mbar_init(wfull_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp == 0) {
    {   // whole warp, converged: see elect_one()
      mbar_expect_tx_e(wfull_bar, (uint32_t)p.w_tx);
      for (int tap = 0; tap < 27; ++tap)          // smem slot order [(kh,kw)][kd = 2,1,0]
        tma_load_2d_e(w_base + ((tap % 9) * 3 + (2 - tap / 9)) * p.w_slab, &map_w, wfull_bar, 0, tap * p.Cout);
      int stage = 0; uint32_t phase = 0;
      for (int item = blockIdx.x; item < p.nitems; item += gridDim.x) {
        int t = item;
        const int seg = t % p.nseg; t /= p.nseg;
        const int x0 = (t % p.ntx) * 8; t /= p.ntx;
        const int y0 = (t % p.nty) * 16; const int n = t / p.nty;
        const int zs = seg * p.lseg;
        const int L = (p.D - zs) < p.lseg ? (p.D - zs) : p.lseg;
        for (int ip = 0; ip < L + 2; ++ip) {
          mbar_wait(empty_bar + 8 * stage, phase ^ 1);
          mbar_expect_tx_e(full_bar + 8 * stage, (uint32_t)p.plane_tx);
          tma_load_5d_e(a_base + stage * p.plane_bytes, &map_x, full_bar + 8 * stage, 0, x0 - 1, y0 - 1, zs - 1 + ip, n);
          if (++stage == p.ring) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {                                             // whole warp, converged; see elect_one()
      mbar_wait(wfull_bar, 0);
      int stage = 0; uint32_t phase = 0; int oc = 0;
      constexpr int KSTEPS = KC / 16;
      constexpr uint32_t ROWB = KC * 2;
      const uint32_t hi_a = desc_hi(p.a_sbo, p.layout_type), hi_b = desc_hi(p.sbo, p.layout_type);
      const uint32_t slab16 = (uint32_t)p.w_slab >> 4, w16 = w_base >> 4;
      // nb is 4 or 8: accumulator slot and phase by mask and shift - an integer division by the runtime nb costs ~20
      // instructions, and this warp's instruction path is the critical path of the plane step (DESIGN.md section 4, finding 9)
      const int nbm = p.nb - 1, nbs = __ffs(p.nb) - 1;
      for (int item = blockIdx.x; item < p.nitems; item += gridDim.x) {
        const int seg = item % p.nseg;
        const int zs = seg * p.lseg;
        const int L = (p.D - zs) < p.lseg ? (p.D - zs) : p.lseg;
        for (int ip = 0; ip < L + 2; ++ip) {
          mbar_wait((XF ? xf_bar : full_bar) + 8 * stage, phase);
          tc_fence_after();
          const uint32_t lo_a = (a_base + stage * p.plane_bytes) >> 4;
          const int kd_hi = ip < 2 ? ip : 2;                      // kd with 0 <= ip - kd < L
          const int kd_lo = ip - (L - 1) > 0 ? ip - (L - 1) : 0;
          const bool fresh = kd_lo == 0;                          // output plane ip receives its first contribution
          if (fresh) { const int ocz = oc + ip; mbar_wait(tempty_bar + 8 * (ocz & nbm), ((ocz >> nbs) & 1) ^ 1); tc_fence_after(); }
          // runs of adjacent accumulators (planes ip-kd for kd = hi..lo ascend; a run ends at the ring wrap or at maxblk)
          uint32_t dA = 0, bA = 0, iA = 0, dB = 0, bB = 0, iB = 0, dC = 0, bC = 0, iC = 0; int nruns = 0;
          for (int kd = kd_hi; kd >= kd_lo;) {
            const int b0 = (oc + ip - kd) & nbm;
            int len = 1;
            while (kd - len >= kd_lo && b0 + len <= nbm && len < p.maxblk) ++len;
            const uint32_t d = tmem_base + (uint32_t)(b0 * p.acc_cols), bo = (uint32_t)(2 - kd) * slab16, id = p.idesc0 | ((uint32_t)len * p.n8) << 17;
            if (nruns == 0) { dA = d; bA = bo; iA = id; } else if (nruns == 1) { dB = d; bB = bo; iB = id; } else { dC = d; bC = bo; iC = id; }
            ++nruns;
            kd -= len;
          }
          // the very first MMA into a fresh plane must overwrite: that plane (kd = 0, the last block) is issued on its own
          const uint32_t dF = tmem_base + (uint32_t)(((oc + ip) & nbm) * p.acc_cols);
          const uint32_t id1 = p.idesc0 | (p.n8 << 17);
#pragma unroll
          for (int kh = 0; kh < 3; ++kh)
#pragma unroll
            for (int kw = 0; kw < 3; ++kw)
#pragma unroll
              for (int k = 0; k < (SPLIT ? KSTEPS / 2 * 3 : KSTEPS); ++k) {
                constexpr int KH = KSTEPS / 2;
                const int ka = SPLIT ? (k < 2 * KH ? k : k - 2 * KH) : k;          // hi, lo, hi
                const int kb = SPLIT ? (k < KH ? k : k - KH) : k;                  // whi, whi, wlo
                const uint32_t da = lo_a + (((kh * 10 + kw) * ROWB + ka * 32) >> 4);
                const uint32_t db = w16 + (uint32_t)((kh * 3 + kw) * 3) * slab16 + ((kb * 32) >> 4);
                if (kh == 0 && kw == 0 && k == 0 && fresh) {
                  tc_mma_f16_e(dF, desc_pack(hi_a, da), desc_pack(hi_b, db + 2 * slab16), id1, 0);
                  for (int kd = kd_hi; kd >= 1; --kd)
                    tc_mma_f16_e(tmem_base + (uint32_t)(((oc + ip - kd) & nbm) * p.acc_cols), desc_pack(hi_a, da),
                               desc_pack(hi_b, db + (uint32_t)(2 - kd) * slab16), id1, 1);
                } else {
                  tc_mma_f16_e(dA, desc_pack(hi_a, da), desc_pack(hi_b, db + bA), iA, 1);
                  if (nruns > 1) tc_mma_f16_e(dB, desc_pack(hi_a, da), desc_pack(hi_b, db + bB), iB, 1);
                  if (nruns > 2) tc_mma_f16_e(dC, desc_pack(hi_a, da), desc_pack(hi_b, db + bC), iC, 1);
                }
              }
          tc_commit_e(empty_bar + 8 * stage);
          if (ip >= 2) tc_commit_e(tfull_bar + 8 * ((oc + ip - 2) & nbm));
          if (++stage == p.ring) { stage = 0; phase ^= 1; }
        }
        oc += L;
      }
    }
  } else if (XF && warp >= 10) {
    // ===== transform: channels [0, xf_nch) of every in-volume voxel of the plane become relu(fma(raw, a, b)), the very
    // expression seg3d_gn_apply evaluates; in place, same swizzled addresses (64-byte rows: 16-byte chunk c of row r sits at
    // chunk c ^ ((r >> 1) & 3)); zero padding stays zero.  A thread owns ONE logical chunk, so its 8 scales / shifts are fixed.
    if constexpr (XF) {
      static_assert(!XF || KC == 32, "the transform stage is written for 64-byte rows");
      const int t = (warp - 10) * 32 + lane;
      const int gch = p.xf_nch >> 3;                  // chunks per row that need the transform (1..4)
      const int c = t % gch, r0 = t / gch, rstep = 128 / gch;
      float sa[8], sb[8];
      int stage = 0; uint32_t phase = 0; int cur_n = -1;
      for (int item = blockIdx.x; item < p.nitems; item += gridDim.x) {
        int tt = item;
        const int seg = tt % p.nseg; tt /= p.nseg;
        const int x0 = (tt % p.ntx) * 8; tt /= p.ntx;
        const int y0 = (tt % p.nty) * 16; const int n = tt / p.nty;
        const int zs = seg * p.lseg;
        const int L = (p.D - zs) < p.lseg ? (p.D - zs) : p.lseg;
        if (n != cur_n) {
          float mean, rstd;
          gn_mean_rstd(p.xf_stats + 2 * n, p.xf_count, p.xf_eps, mean, rstd);
#pragma unroll
          for (int j = 0; j < 8; ++j) { sa[j] = rstd * p.xf_gamma[8 * c + j]; sb[j] = p.xf_beta[8 * c + j] - mean * sa[j]; }
          cur_n = n;
        }
        for (int ip = 0; ip < L + 2; ++ip) {
          mbar_wait(full_bar + 8 * stage, phase);
          const int gz = zs - 1 + ip;
          if (gz >= 0 && gz < p.D && r0 < rstep) {
            uint8_t* plane = smem_al + 27 * p.w_slab + stage * p.plane_bytes;
            for (int r = r0; r < 180; r += rstep) {
              const int hy = r / 10, hx = r - hy * 10;
              const int gx = x0 - 1 + hx, gy = y0 - 1 + hy;
              if (gx < 0 || gx >= p.W || gy < 0 || gy >= p.H) continue;
              T* slot = reinterpret_cast<T*>(plane + r * 64 + ((c ^ ((r >> 1) & 3)) << 4));
              Vec8<T> v; v.load(slot);
              float f[8]; v.get(f);
#pragma unroll
              for (int j = 0; j < 8; ++j) f[j] = fmaxf(fmaf(f[j], sa[j], sb[j]), 0.f);
              v.set(f); v.store(slot);
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(xf_bar + 8 * stage);
          if (++stage == p.ring) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;             // warps 2-5: even 16-column chunks, warps 6-9: odd ones
    const int r = q * 32 + lane;
    const int lx = r & 7, ly = r >> 3;
    float s = 0.f, ss = 0.f;
    int cur_n = -1, oc = 0;
    const bool wide = p.wide != 0;
    for (int item = blockIdx.x; item < p.nitems; item += gridDim.x) {
      int t = item;
      const int seg = t % p.nseg; t /= p.nseg;
      const int x0 = (t % p.ntx) * 8; t /= p.ntx;
      const int y0 = (t % p.nty) * 16; const int n = t / p.nty;
      const int zs = seg * p.lseg;
      const int L = (p.D - zs) < p.lseg ? (p.D - zs) : p.lseg;
      if (stats && n != cur_n) {
        if (cur_n >= 0) {
          s = warp_sum(s); ss = warp_sum(ss);
          if (lane == 0) { atomicAdd(stats + 2 * cur_n, (double)s); atomicAdd(stats + 2 * cur_n + 1, (double)ss); }
        }
        s = 0.f; ss = 0.f; cur_n = n;
      }
      const int gx = x0 + lx, gy = y0 + ly;
      const bool valid = (gx < p.W) && (gy < p.H);
      for (int zl = 0; zl < L; ++zl) {
        const int ocz = oc + zl, buf = ocz & (p.nb - 1);           // nb is 4 or 8
        const size_t vox = (((size_t)n * p.D + (zs + zl)) * p.H + gy) * p.W + gx;
        T* yrow = y + vox * p.y_ld;
        float* yrow32 = reinterpret_cast<float*>(y) + vox * p.y_ld;
        mbar_wait(tfull_bar + 8 * buf, (ocz >> (__ffs(p.nb) - 1)) & 1);
        tc_fence_after();
        const uint32_t tcol = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * p.acc_cols);
        for (int c0 = half * 16; c0 < p.Cout; c0 += 32) {
          uint32_t v[16];
          tc_ld16(tcol + (uint32_t)c0, v);
          tc_wait_ld();
          float f[16];
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) {
            f[jj] = __uint_as_float(v[jj]) + (bias ? bias[c0 + jj] : 0.f);
            if (valid) { s += f[jj]; ss += f[jj] * f[jj]; }
          }
          if (valid) {
            if (p.out_f32 == 2) {      // fp32 rows of pitch y_ld >= Cout (16-byte aligned): split mode
              float4* d4 = reinterpret_cast<float4*>(yrow32 + c0);
#pragma unroll
              for (int jj = 0; jj < 16; jj += 4) d4[jj >> 2] = make_float4(f[jj], f[jj + 1], f[jj + 2], f[jj + 3]);
            } else if (p.out_f32) {    // only the first y_ld (= real) channels are kept, densely packed
#pragma unroll
              for (int jj = 0; jj < 16; ++jj) if (c0 + jj < p.y_ld) yrow32[c0 + jj] = f[jj];
            } else {
              store16<T>(yrow + c0, f, wide);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar + 8 * buf);
      }
      oc += L;
    }
    if (stats && cur_n >= 0) {
      s = warp_sum(s); ss = warp_sum(ss);
      if (lane == 0) { atomicAdd(stats + 2 * cur_n, (double)s); atomicAdd(stats + 2 * cur_n + 1, (double)ss); }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}


// ---------------------------------------------------------------------------------------------------
// Weight gradient of the k3 convolution on the tensor cores:
//     dW[tap][ci][co] = sum over voxels v of  dy[v][co] * x[v + tap][ci]
// is a GEMM with K = voxels.  Both operands are stored voxel-major with the channels contiguous, i.e.
// they are MN-major UMMA operands exactly as the TMA delivers them (128B/64B/32B swizzled rows):
//     A = dy^T : M = co (128 rows of TMEM, zero / don't-care beyond Cout), K = the 128 voxels of an 8x16 plane tile
//     B = x    : N = ci block (<= 64), K = the same voxels shifted by (kh,kw) inside a 10x18 halo plane
// A CTA owns one (co block, ci block, tap group) and accumulates its D_tap[co][ci] tiles in TMEM over all the
// voxel tiles of its K split (persistent), then adds them to the fp32 gradient with coalesced atomics.
// Tap group = one kd (9 taps) for N <= 32, one (kd,kh) (3 taps) for N = 64, so the x plane needed with dy plane z
// is the single plane z+kd-1: a two-operand TMA pipeline, no plane ring.
struct WgParams {
  int Cin, Cout, nblk, mblk;            // N (ci) block width, M (co) block width (<=128)
  int n_ci_blk, n_co_blk, ngroups, taps_per_group;
  int D, H, W, N, ntx, nty, ntiles;     // tiles over (n, z, ty, tx)
  int stages, a_bytes, b_bytes, a_tx, b_tx, a_atoms;
  int b_row_bytes;
  int tmem_cols;
  int merge_kw;
  uint32_t idesc, idesc3, a_sbo, a_lbo, b_sbo, a_layout, b_layout;
};

template <typename T, int NBLK, int TPG>
__global__ void __launch_bounds__(TC_THREADS)
conv3d_k3_wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x,
                          const WgParams p, float* __restrict__ dw) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t a_base = smem_base;
  const uint32_t b_base = smem_base + p.stages * p.a_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_al + p.stages * (p.a_bytes + p.b_bytes));
  const uint32_t full_bar = smem_u32(bars);
  const uint32_t empty_bar = full_bar + 8 * p.stages;
  const uint32_t done_bar = empty_bar + 8 * p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * p.stages + 1);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler

  // blockIdx.y -> (co block, ci block, tap group)
  int c = blockIdx.y;
  const int grp = c % p.ngroups; c /= p.ngroups;
  const int cib = c % p.n_ci_blk; const int cob = c / p.n_ci_blk;
  const int kd = p.taps_per_group == 9 ? grp : grp / 3;
  const int kh0 = p.taps_per_group == 9 ? 0 : grp % 3;          // first kh of the group
  const int ci0 = cib * p.nblk, co0 = cob * p.mblk;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_dy) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    for (int s = 0; s < p.stages; ++s) { mbar_init(full_bar + 8 * s, 1); mbar_init(empty_bar + 8 * s, 1); }
    mbar_init(done_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp == 0) {
    {   // whole warp, converged: see elect_one()
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        int t = tile;
        const int x0 = (t % p.ntx) * 8; t /= p.ntx;
        const int y0 = (t % p.nty) * 16; t /= p.nty;
        const int z = t % p.D; const int n = t / p.D;
        mbar_wait(empty_bar + 8 * stage, phase ^ 1);
        mbar_expect_tx_e(full_bar + 8 * stage, (uint32_t)(p.a_tx + p.b_tx));
        for (int a = 0; a < p.a_atoms; ++a)
          tma_load_5d_e(a_base + stage * p.a_bytes + a * 16384, &map_dy, full_bar + 8 * stage, co0 + a * 64, x0, y0, z, n);
        tma_load_5d_e(b_base + stage * p.b_bytes, &map_x, full_bar + 8 * stage, ci0, x0 - 1, y0 - 1, z + kd - 1, n);
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    {   // whole warp, converged: see elect_one()
      int stage = 0; uint32_t phase = 0;
      const uint32_t hi_a = desc_hi(p.a_sbo, p.a_layout), hi_b = desc_hi(p.b_sbo, p.b_layout);
      const uint32_t lbo_a = ((p.a_lbo >> 4) & 0x3FFFu) << 16;
      constexpr uint32_t RB16 = (NBLK * 2) >> 4;               // halo row bytes / 16
      constexpr uint32_t KSTEP_B = (2 * 10 * NBLK * 2) >> 4;   // two x-lines of the halo per K=16 step
      const uint32_t kh_off = (uint32_t)(kh0 * 10) * RB16;
      uint32_t accumulate = 0;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        mbar_wait(full_bar + 8 * stage, phase);
        tc_fence_after();
        const uint32_t lo_a = ((a_base + stage * p.a_bytes) >> 4) | lbo_a;
        const uint32_t lo_b0 = ((b_base + stage * p.b_bytes) >> 4) + kh_off;
        // one MMA covers the three kw taps of a kh row: N = 3*NBLK, the three N-atoms of the MN-major B operand are
        // the same halo rows shifted by one voxel each (LBO = one row), so A is read once per kh instead of per tap
        if (p.merge_kw) {
#pragma unroll
          for (int khi = 0; khi < TPG / 3; ++khi) {
            const uint32_t lo_b = (lo_b0 + (uint32_t)(khi * 10) * RB16) | (RB16 << 16);
            const uint32_t dcol = tmem_base + (uint32_t)(khi * 3 * NBLK);
#pragma unroll
            for (int k = 0; k < 8; ++k)
              tc_mma_f16_e(dcol, desc_pack(hi_a, lo_a + (uint32_t)((k * 2048) >> 4)), desc_pack(hi_b, lo_b + (uint32_t)k * KSTEP_B),
                         p.idesc3, k == 0 ? accumulate : 1u);
          }
        } else {
#pragma unroll
          for (int tg = 0; tg < TPG; ++tg) {
            const uint32_t lo_b = lo_b0 + (uint32_t)((tg / 3) * 10 + tg % 3) * RB16;
            const uint32_t dcol = tmem_base + (uint32_t)(tg * NBLK);
#pragma unroll
            for (int k = 0; k < 8; ++k)      // 128 voxels = 8 steps of K=16 (two 8-voxel x-lines each)
              tc_mma_f16_e(dcol, desc_pack(hi_a, lo_a + (uint32_t)((k * 2048) >> 4)), desc_pack(hi_b, lo_b + (uint32_t)k * KSTEP_B),
                         p.idesc, k == 0 ? accumulate : 1u);
          }
        }
        accumulate = 1;
        tc_commit_e(empty_bar + 8 * stage);
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
      tc_commit_e(done_bar);
    }
  } else {
    // epilogue (once): TMEM lane = co, column = (tap in group, ci)
    const int q = warp & 3;
    const int co = q * 32 + lane;
    mbar_wait(done_bar, 0);
    tc_fence_after();
    const bool has_tiles = blockIdx.x < p.ntiles;
    if (has_tiles) {
      for (int tg = 0; tg < p.taps_per_group; ++tg) {
        const int tap = (kd * 3 + kh0 + tg / 3) * 3 + tg % 3;
        for (int c0 = 0; c0 < p.nblk; c0 += 16) {
          uint32_t v[16];
          tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(tg * p.nblk + c0), v);
          tc_wait_ld();
          if (co < p.mblk && co0 + co < p.Cout) {
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
              const int ci = ci0 + c0 + jj;
              if (ci < p.Cin) atomicAdd(dw + ((size_t)tap * p.Cin + ci) * p.Cout + co0 + co, __uint_as_float(v[jj]));
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}


// Weight gradient of the stride-2 convolutions on the tensor cores (same scheme as the k3 kernel above):
//   MODE 1 (k2 s2 down-conv)    dW[tap][ci][co] = sum_vo x[2vo+tap][ci] * dy[vo][co]   A = dy tile, B_tap = x through the folded-stride map
//   MODE 2 (transposed up-conv) dW[ci][tap*Cout+co] = sum_v x[v][ci] * dy[2v+tap][co]  A_tap = dy through the folded-stride map, B = x tile
// A CTA owns (co block, ci block, (kd,kh)) and the two kw taps; K tiles are 8x16 planes of the low-resolution grid.
struct Wg2Params {
  int mode, Cin, Cout, nblk, mblk, n_ci_blk, n_co_blk;
  int D, H, W, N, ntx, nty, ntiles;          // low-resolution grid (dy for MODE 1, x for MODE 2)
  int fold_ld, foldW, foldH;                 // folded tensor: channel pitch and the low-res W, H used in the coordinate folding
  int stages, a_bytes, b_bytes, a_slab, b_slab, tx_bytes, a_atoms, b_row_bytes, tmem_cols;
  uint32_t idesc, b_sbo, b_layout;
};

template <typename T, int NBLK, int MODE>
__global__ void __launch_bounds__(TC_THREADS)
conv3d_s2_wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x,
                          const Wg2Params p, float* __restrict__ dw) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t a_base = smem_base;
  const uint32_t b_base = smem_base + p.stages * p.a_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_al + p.stages * (p.a_bytes + p.b_bytes) + 16384);
  const uint32_t full_bar = smem_u32(bars);
  const uint32_t empty_bar = full_bar + 8 * p.stages;
  const uint32_t done_bar = empty_bar + 8 * p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * p.stages + 1);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler
  int c = blockIdx.y;
  const int grp = c & 3; c >>= 2;
  const int cib = c % p.n_ci_blk; const int cob = c / p.n_ci_blk;
  const int kd = grp >> 1, kh = grp & 1;
  const int ci0 = cib * p.nblk, co0 = cob * p.mblk;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_dy) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    for (int s = 0; s < p.stages; ++s) { mbar_init(full_bar + 8 * s, 1); mbar_init(empty_bar + 8 * s, 1); }
    mbar_init(done_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp == 0) {
    {   // whole warp, converged: see elect_one()
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        int t = tile;
        const int x0 = (t % p.ntx) * 8; t /= p.ntx;
        const int y0 = (t % p.nty) * 16; t /= p.nty;
        const int z = t % p.D; const int n = t / p.D;
        mbar_wait(empty_bar + 8 * stage, phase ^ 1);
        const uint32_t fb = full_bar + 8 * stage, sa = a_base + stage * p.a_bytes, sb = b_base + stage * p.b_bytes;
        mbar_expect_tx_e(fb, (uint32_t)p.tx_bytes);
        if (MODE == 1) {
          for (int a = 0; a < p.a_atoms; ++a) tma_load_5d_e(sa + a * 16384, &map_dy, fb, co0 + a * 64, x0, y0, z, n);
          for (int kw = 0; kw < 2; ++kw)
            tma_load_5d_e(sb + kw * p.b_slab, &map_x, fb, kw * p.fold_ld + ci0, x0 + kh * p.foldW, y0 + kd * p.foldH, z, n);
        } else {
          for (int kw = 0; kw < 2; ++kw)
            for (int a = 0; a < p.a_atoms; ++a)
              tma_load_5d_e(sa + kw * p.a_slab + a * 16384, &map_dy, fb, kw * p.fold_ld + co0 + a * 64, x0 + kh * p.foldW, y0 + kd * p.foldH, z, n);
          tma_load_5d_e(sb, &map_x, fb, ci0, x0, y0, z, n);
        }
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    {   // whole warp, converged: see elect_one()
      int stage = 0; uint32_t phase = 0;
      const uint32_t hi_a = desc_hi(1024, 2), hi_b = desc_hi(p.b_sbo, p.b_layout);
      const uint32_t lbo_a = ((16384u >> 4) & 0x3FFFu) << 16;
      constexpr uint32_t KSTEP_B = (16 * NBLK * 2) >> 4;       // 16 dense rows per K=16 step
      const uint32_t a_slab16 = (uint32_t)p.a_slab >> 4, b_slab16 = (uint32_t)p.b_slab >> 4;
      uint32_t accumulate = 0;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        mbar_wait(full_bar + 8 * stage, phase);
        tc_fence_after();
        const uint32_t lo_a0 = ((a_base + stage * p.a_bytes) >> 4) | lbo_a;
        const uint32_t lo_b0 = (b_base + stage * p.b_bytes) >> 4;
#pragma unroll
        for (int kw = 0; kw < 2; ++kw) {
          const uint32_t lo_a = lo_a0 + (MODE == 2 ? kw * a_slab16 : 0u);
          const uint32_t lo_b = lo_b0 + (MODE == 1 ? kw * b_slab16 : 0u);
          const uint32_t dcol = tmem_base + (uint32_t)(kw * NBLK);
#pragma unroll
          for (int k = 0; k < 8; ++k)
            tc_mma_f16_e(dcol, desc_pack(hi_a, lo_a + (uint32_t)((k * 2048) >> 4)), desc_pack(hi_b, lo_b + (uint32_t)k * KSTEP_B),
                       p.idesc, k == 0 ? accumulate : 1u);
        }
        accumulate = 1;
        tc_commit_e(empty_bar + 8 * stage);
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
      tc_commit_e(done_bar);
    }
  } else {
    const int q = warp & 3;
    const int co = q * 32 + lane;
    mbar_wait(done_bar, 0);
    tc_fence_after();
    for (int kw = 0; kw < 2; ++kw) {
      const int tap = (kd * 2 + kh) * 2 + kw;
      for (int c0 = 0; c0 < NBLK; c0 += 16) {
        uint32_t v[16];
        tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(kw * NBLK + c0), v);
        tc_wait_ld();
        if (co < p.mblk && co0 + co < p.Cout) {
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) {
            const int ci = ci0 + c0 + jj;
            if (ci < p.Cin) {
              const size_t o = MODE == 1 ? ((size_t)tap * p.Cin + ci) * p.Cout + co0 + co : ((size_t)ci * 8 + tap) * p.Cout + co0 + co;
              atomicAdd(dw + o, __uint_as_float(v[jj]));
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}

// ---- host side -----------------------------------------------------------------------------------
template <typename T>
cudaError_t launch_tc(dim3 grid, size_t smem, cudaStream_t st, const CUtensorMap& mx, const CUtensorMap& mw,
                      const TcParams& p, const float* bias, void* y, double* stats) {
  cudaError_t e;
#define SEG3D_LAUNCH_P(KCV)                                                                                              \
  e = cudaFuncSetAttribute(conv3d_tc_persistent_kernel<T, KCV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
  if (e != cudaSuccess) return e;                                                                                        \
  conv3d_tc_persistent_kernel<T, KCV><<<grid, TCE_THREADS, smem, st>>>(mx, mw, p, bias, (T*)y, stats);
  if (p.KC == 64) { SEG3D_LAUNCH_P(64) } else if (p.KC == 32) { SEG3D_LAUNCH_P(32) } else { SEG3D_LAUNCH_P(16) }
#undef SEG3D_LAUNCH_P
  return cudaGetLastError();
}

}  // namespace

int seg3d_conv_tc_supported(int mode, int dtype, int Cin, int Cout, int x_ld, int y_ld, int D, int H, int W) {
  const int out_f32 = dtype & SEG3D_OUT_F32;
  dtype &= ~SEG3D_OUT_F32;
  if (mode != SEG3D_CONV_K3 && mode != SEG3D_CONV_K2S2 && mode != SEG3D_CONV_T2S2) return 0;
  if (dtype != SEG3D_F16 && dtype != SEG3D_BF16) return 0;
  if (Cin % 16 || Cout % 16 || Cout > 256 || Cin > 1024) return 0;
  if (x_ld % 8 || (!out_f32 && y_ld % 8)) return 0;
  if (out_f32 && !(mode == SEG3D_CONV_K3 && (Cin == 16 || Cin == 32 || Cin == 64) && W % 8 == 0 && D >= 4)) return 0;
  if (mode == SEG3D_CONV_K2S2 && (D % 2 || H % 2 || W % 2)) return 0;
  return 1;
}

int seg3d_conv_tc(int mode, int dtype, const void* x, int x_ld, int Cin, const void* w, const float* bias,
                  void* y, int y_ld, int Cout, int N, int D, int H, int W, double* stats, cudaStream_t st,
                  int epi_mode, const double* gn_stats, const float* gn_gamma, const float* gn_beta, float gn_eps,
                  int split_lo_off, int out_f32_generic,
                  int xf_nch, const double* xf_stats, const float* xf_gamma, const float* xf_beta, float xf_eps) {
  EncodeTiledFn encode = get_encode();
  if (!encode) { seg3d_set_error("conv_tc: cuTensorMapEncodeTiled entry point not available"); return SEG3D_ECUDA; }
  SEG3D_REQUIRE(((uintptr_t)x) % 16 == 0 && ((uintptr_t)w) % 16 == 0 && ((uintptr_t)y) % 16 == 0, "conv_tc: pointers must be 16-byte aligned");

  // ---- z-marching kernel for narrow k3 layers --------------------------------------------------------
  const int out_f32 = (dtype & SEG3D_OUT_F32) ? 1 : 0;
  dtype &= ~SEG3D_OUT_F32;
  // split operands take the z-march kernel when the lo half follows the hi half directly (rows [hi(Cin) | lo(Cin)]): the row is
  // then one K block of 2*Cin channels
  const bool zm_split = split_lo_off > 0 && split_lo_off == Cin && out_f32_generic && (Cin == 16 || Cin == 32) && y_ld % 4 == 0 &&
                        dtype == SEG3D_F16 && env_int("SEG3D_ZM_SPLIT", 1) != 0;
  if (epi_mode == 0 && ((split_lo_off == 0 && !out_f32_generic && (Cin == 16 || Cin == 32 || Cin == 64)) || zm_split) && mode == SEG3D_CONV_K3 && W % 8 == 0 && D >= 4 && env_int("SEG3D_TC_ZMARCH", 1) != 0) {
    ZmParams z;
    memset(&z, 0, sizeof(z));
    const int Cin_real = Cin;
    if (zm_split) Cin = 2 * Cin;                       // the K block: [hi | lo] channels of a row, [whi | wlo] of a weight row
    z.Cout = Cout; z.KC = Cin; z.row_bytes = Cin * 2;
    z.D = D; z.H = H; z.W = W; z.N = N; z.y_ld = y_ld; z.out_f32 = zm_split ? 2 : out_f32;
    z.xf_nch = xf_nch; z.xf_stats = xf_stats; z.xf_gamma = xf_gamma; z.xf_beta = xf_beta; z.xf_eps = xf_eps;
    z.xf_count = (double)xf_nch * D * H * W;
    z.wide = (!out_f32 && wide_ok(y, y_ld, 2) && env_int("SEG3D_WIDE_ST", 1)) ? 1 : 0;
    z.w_slab = (Cout * z.row_bytes + 1023) & ~1023;
    z.plane_tx = 180 * z.row_bytes;
    z.plane_bytes = (z.plane_tx + 1023) & ~1023;
    z.w_tx = 27 * Cout * z.row_bytes;
    if (27 * z.w_slab <= 112 * 1024) {
      z.ntx = W / 8; z.nty = (H + 15) / 16;
      z.acc_cols = Cout <= 16 ? 16 : (Cout <= 32 ? 32 : 64);
      z.nb = z.acc_cols <= 32 ? 8 : 4;
      z.tmem_cols = z.nb * z.acc_cols;
      // one MMA may span up to three adjacent accumulators when every weight slab is a whole number of 1024-byte swizzle
      // repeats (so the [(kh,kw)][kd] slabs are contiguous) and the accumulator pitch equals Cout
      z.maxblk = (z.w_slab == Cout * z.row_bytes && z.acc_cols == Cout && 3 * Cout <= 256) ? env_int("SEG3D_ZM_MAXBLK", 3) : 1;
      if (z.maxblk < 1) z.maxblk = 1;
      if (z.maxblk > 3) z.maxblk = 3;
      int ctas_per_sm = env_int("SEG3D_ZM_CTAS_PER_SM", 2);
      if (ctas_per_sm * z.tmem_cols > 512) ctas_per_sm = 512 / z.tmem_cols;
      int ring = ((200 * 1024 / ctas_per_sm) - 27 * z.w_slab) / z.plane_bytes;
      if (ring < 3) { ctas_per_sm = 1; ring = (200 * 1024 - 27 * z.w_slab) / z.plane_bytes; }
      if (ring > 8) ring = 8;
      { const int e = env_int("SEG3D_ZM_RING", 0); if (e >= 2) ring = e; }
      z.ring = ring;
      // z segments: enough work items to balance ~4 per resident CTA, halo overhead 2/lseg
      const long long cols = (long long)N * z.ntx * z.nty;
      const long long want = 4ll * ctas_per_sm * seg3d_num_sms();
      int nseg = (int)((want + cols - 1) / cols);
      if (nseg < 1) nseg = 1;
      int lseg = (D + nseg - 1) / nseg;
      if (lseg < 8) lseg = D < 8 ? D : 8;
      { const int e = env_int("SEG3D_ZM_LSEG", 0); if (e >= 1) lseg = e; }
      z.lseg = lseg; z.nseg = (D + lseg - 1) / lseg;
      const long long nitems = cols * z.nseg;
      if (ring >= 3 && nitems < (1ll << 31)) {
        z.nitems = (int)nitems;
        z.sbo = 8 * z.row_bytes; z.a_sbo = 10 * z.row_bytes;
        z.layout_type = z.row_bytes == 128 ? 2u : (z.row_bytes == 64 ? 4u : 6u);
        const uint32_t fmt = dtype == SEG3D_BF16 ? 1u : 0u;
        z.idesc0 = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(TILE_M >> 4) << 24);
        z.n8 = (uint32_t)(Cout >> 3);
        const CUtensorMapDataType tdt = dtype == SEG3D_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
        const CUtensorMapSwizzle sw = z.row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (z.row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
        CUtensorMap map_x, map_w;
        cuuint64_t dims[5] = {(cuuint64_t)Cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)N};
        cuuint64_t strides[4] = {(cuuint64_t)x_ld * 2, (cuuint64_t)W * x_ld * 2, (cuuint64_t)H * W * x_ld * 2, (cuuint64_t)D * H * W * x_ld * 2};
        cuuint32_t box[5] = {(cuuint32_t)Cin, 10, 18, 1, 1};
        cuuint32_t estr[5] = {1, 1, 1, 1, 1};
        CUresult r = encode(&map_x, tdt, 5, const_cast<void*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { seg3d_set_error("conv_tc(zmarch): cuTensorMapEncodeTiled(x) failed with %d", (int)r); return SEG3D_ECUDA; }
        cuuint64_t wdims[2] = {(cuuint64_t)Cin, (cuuint64_t)27 * Cout};
        cuuint64_t wstr[1] = {(cuuint64_t)Cin * 2};
        cuuint32_t wbox[2] = {(cuuint32_t)Cin, (cuuint32_t)Cout};
        cuuint32_t westr[2] = {1, 1};
        r = encode(&map_w, tdt, 2, const_cast<void*>(w), wdims, wstr, wbox, westr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { seg3d_set_error("conv_tc(zmarch): cuTensorMapEncodeTiled(w) failed with %d", (int)r); return SEG3D_ECUDA; }
        const size_t smem = 1024 + (size_t)27 * z.w_slab + (size_t)ring * z.plane_bytes + (3 * ring + 2 * ZM_MAXNB + 1) * 8 + 64;
        const long long max_grid = (long long)ctas_per_sm * seg3d_num_sms();
        dim3 grid((unsigned)(nitems < max_grid ? nitems : max_grid));
        cudaError_t e = cudaSuccess;
#define SEG3D_LAUNCH_Z(TT, KCV)                                                                                             \
        { e = cudaFuncSetAttribute(conv3d_k3_zmarch_kernel<TT, KCV, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  \
          if (e == cudaSuccess) { conv3d_k3_zmarch_kernel<TT, KCV, false><<<grid, TCE_THREADS, smem, st>>>(map_x, map_w, z, bias, (TT*)y, stats); e = cudaGetLastError(); } }
#define SEG3D_LAUNCH_ZS(KCV)                                                                                                \
        { e = cudaFuncSetAttribute(conv3d_k3_zmarch_kernel<__half, KCV, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  \
          if (e == cudaSuccess) { conv3d_k3_zmarch_kernel<__half, KCV, true><<<grid, TCE_THREADS, smem, st>>>(map_x, map_w, z, bias, (__half*)y, stats); e = cudaGetLastError(); } }
        if (xf_nch > 0) {          // GroupNorm + ReLU of the first xf_nch input channels formed in shared memory (64-byte rows only)
          if (zm_split || Cin != 32 || (xf_nch != 8 && xf_nch != 16 && xf_nch != 32) || !xf_stats || !xf_gamma || !xf_beta) {
            seg3d_set_error("conv_tc(zmarch): the input transform needs Cin == 32 and 8, 16 or 32 transformed channels");
            return SEG3D_EUNSUPPORTED;
          }
          if (dtype == SEG3D_BF16) {
            e = cudaFuncSetAttribute(conv3d_k3_zmarch_kernel<__nv_bfloat16, 32, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e == cudaSuccess) { conv3d_k3_zmarch_kernel<__nv_bfloat16, 32, false, true><<<grid, ZMX_THREADS, smem, st>>>(map_x, map_w, z, bias, (__nv_bfloat16*)y, stats); e = cudaGetLastError(); }
          } else {
            e = cudaFuncSetAttribute(conv3d_k3_zmarch_kernel<__half, 32, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e == cudaSuccess) { conv3d_k3_zmarch_kernel<__half, 32, false, true><<<grid, ZMX_THREADS, smem, st>>>(map_x, map_w, z, bias, (__half*)y, stats); e = cudaGetLastError(); }
          }
        } else if (zm_split) {
          if (Cin == 64) SEG3D_LAUNCH_ZS(64) else SEG3D_LAUNCH_ZS(32)
        } else if (dtype == SEG3D_BF16) {
          if (Cin == 64) SEG3D_LAUNCH_Z(__nv_bfloat16, 64) else if (Cin == 32) SEG3D_LAUNCH_Z(__nv_bfloat16, 32) else SEG3D_LAUNCH_Z(__nv_bfloat16, 16)
        } else {
          if (Cin == 64) SEG3D_LAUNCH_Z(__half, 64) else if (Cin == 32) SEG3D_LAUNCH_Z(__half, 32) else SEG3D_LAUNCH_Z(__half, 16)
        }
#undef SEG3D_LAUNCH_Z
#undef SEG3D_LAUNCH_ZS
        if (e != cudaSuccess) { seg3d_set_error("conv3d_k3_zmarch_kernel launch failed: %s", cudaGetErrorString(e)); return SEG3D_ECUDA; }
        return SEG3D_OK;
      }
    }
    Cin = Cin_real;            // the shape did not fit the z-march kernel: generic path below
  }
  if (xf_nch > 0) { seg3d_set_error("conv_tc: the input transform is only available on the z-march k3 path (Cin 32, W %% 8 == 0, D >= 4)"); return SEG3D_EUNSUPPORTED; }

  SEG3D_REQUIRE(!out_f32, "conv_tc: SEG3D_OUT_F32 (dense real channels) is only available on the z-march k3 path");
  TcParams p;
  memset(&p, 0, sizeof(p));
  p.conv = mode == SEG3D_CONV_K2S2 ? 1 : (mode == SEG3D_CONV_T2S2 ? 2 : 0);
  const int Do = p.conv == 1 ? D / 2 : D, Ho = p.conv == 1 ? H / 2 : H, Wo = p.conv == 1 ? W / 2 : W;   // GEMM row space
  p.cout_real = Cout; p.npass = 1;
  if (p.conv == 2) {                 // GEMM N = 8*Cout in passes of <= 256 columns
    const int ntot = 8 * Cout;
    const int npc = ntot < 256 ? ntot : 256;
    p.npass = ntot / npc;
    Cout = npc;
  }
  p.Cin = Cin; p.Cout = Cout; p.D = Do; p.H = Ho; p.W = Wo; p.N = N; p.y_ld = y_ld;
  p.x_ld = x_ld; p.halfW = W / 2; p.halfH = H / 2;
  p.wide = (!out_f32_generic && wide_ok(y, y_ld, 2) && p.cout_real % 16 == 0 && env_int("SEG3D_WIDE_ST", 1)) ? 1 : 0;
  p.epi_mode = epi_mode; p.gn_eps = gn_eps; p.gn_stats = gn_stats; p.gn_gamma = gn_gamma; p.gn_beta = gn_beta;
  {
    const long long ovox = p.conv == 1 ? (long long)(D / 2) * (H / 2) * (W / 2) : (p.conv == 2 ? 8ll * D * H * W : (long long)D * H * W);
    p.gn_count = (double)ovox * (double)p.cout_real;
  }
  p.KC = (Cin % 64 == 0) ? 64 : (Cin % 32 == 0 ? 32 : 16);
  p.nchunk_real = Cin / p.KC;
  p.split = split_lo_off > 0 ? 1 : 0; p.lo_off = split_lo_off; p.out_f32 = out_f32_generic;
  p.nchunk = p.split ? 3 * p.nchunk_real : p.nchunk_real;
  const int row_bytes = p.KC * 2;
  p.row_bytes = row_bytes;

  // kw-fused variant (k3 only): one (tw+2)-wide box per (kd,kh) serves the three kw taps through x-shifted
  // descriptors (the swizzle is a function of the absolute smem address, so any row-aligned start works).
  // Needs tw == 8 (every 8-row MMA group is one x-line of the box) and pays 3 weight slabs per stage.
  {
    const int env = env_int("SEG3D_TC_KWFUSE", 2);
    const int slab = (Cout * row_bytes + 1023) & ~1023;
    const bool fits = (10 * 16 * row_bytes + 3 * slab) <= 48 * 1024;
    p.kwfuse = (p.conv == 0 && Wo % 8 == 0 && fits && (env == 1 || (env == 2 && g_kwfuse_default))) ? 1 : 0;
  }
  // tile box: power-of-two dims with product 128 minimising the tile count
  long long best = -1; p.tw = 8; p.th = 4; p.td = 4;
  for (int tw = (p.kwfuse ? 8 : 1); tw <= (p.kwfuse ? 8 : 32); tw *= 2)
    for (int th = 1; th <= 128 / tw; th *= 2) {
      const int td = 128 / (tw * th);
      const long long tiles = (long long)((Wo + tw - 1) / tw) * ((Ho + th - 1) / th) * ((Do + td - 1) / td);
      const long long spread = (tw > 16 || th > 16 || td > 16) ? 512 : 0;      // keep the box compact
      const long long sc = tiles * 1024 - tw * 8 - th + spread;                 // fewer tiles, then wider x, then wider y
      if (best < 0 || sc < best) { best = sc; p.tw = tw; p.th = th; p.td = td; }
    }
  p.ntx = (Wo + p.tw - 1) / p.tw; p.nty = (Ho + p.th - 1) / p.th; p.ntz = (Do + p.td - 1) / p.td;
  const long long ntiles = (long long)p.ntx * p.nty * p.ntz * N * p.npass;
  SEG3D_REQUIRE(ntiles > 0 && ntiles < (1ll << 31), "conv_tc: tile count out of range");
  p.ntiles = (int)ntiles;
  p.ntaps = p.conv == 1 ? 8 : (p.conv == 2 ? 1 : (p.kwfuse ? 9 : 27));

  const int a_rows = p.kwfuse ? (p.tw + 2) * p.th * p.td : TILE_M;
  p.a_bytes = (a_rows * row_bytes + 1023) & ~1023;
  p.b_slab = (Cout * row_bytes + 1023) & ~1023;     // every operand slab stays 1024-byte aligned
  p.b_bytes = p.kwfuse ? 3 * p.b_slab : p.b_slab;
  p.tx_bytes = a_rows * row_bytes + (p.kwfuse ? 3 : 1) * Cout * row_bytes;
  const int stage_bytes = p.a_bytes + p.b_bytes;
  p.sbo = 8 * row_bytes;
  p.a_sbo = p.kwfuse ? (p.tw + 2) * row_bytes : 8 * row_bytes;
  p.layout_type = row_bytes == 128 ? 2u : (row_bytes == 64 ? 4u : 6u);
  const uint32_t fmt = dtype == SEG3D_BF16 ? 1u : 0u;
  p.idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(Cout >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);

  int stages, ctas_per_sm = 1;
  p.acc_cols = Cout <= 16 ? 16 : (Cout <= 32 ? 32 : (Cout <= 64 ? 64 : (Cout <= 128 ? 128 : 256)));
  p.tmem_cols = 2 * p.acc_cols;
  ctas_per_sm = 512 / p.tmem_cols; if (ctas_per_sm > 2) ctas_per_sm = 2;
  ctas_per_sm = env_int("SEG3D_TC_CTAS_PER_SM", ctas_per_sm);
  if (ctas_per_sm * p.tmem_cols > 512) ctas_per_sm = 512 / p.tmem_cols;
  if (ctas_per_sm < 1) ctas_per_sm = 1;
  stages = (200 * 1024 / ctas_per_sm) / stage_bytes;
  if (stages > 8) stages = 8;
  { const int e = env_int("SEG3D_TC_STAGES", 0); if (e >= 2 && e * stage_bytes <= 200 * 1024) stages = e; }
  SEG3D_REQUIRE(stages >= 2, "conv_tc: operand ring does not fit in shared memory (stage %d bytes)", stage_bytes);
  p.stages = stages;

  const CUtensorMapDataType tdt = dtype == SEG3D_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const CUtensorMapSwizzle sw = row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  CUtensorMap map_x, map_w;
  {
    cuuint64_t dims[5], strides[4];
    const int cext = Cin + (p.split ? p.lo_off : 0);      // channel extent the K loop addresses (lo half = +lo_off)
    if (p.conv == 1) {   // stride-2 taps folded into the coordinates: c' = kw*ld + c, x' = x + kh*W/2, y' = y + kd*H/2
      dims[0] = (cuuint64_t)x_ld + cext; dims[1] = (cuuint64_t)W; dims[2] = (cuuint64_t)H; dims[3] = (cuuint64_t)D / 2; dims[4] = (cuuint64_t)N;
      strides[0] = (cuuint64_t)2 * x_ld * 2; strides[1] = (cuuint64_t)2 * W * x_ld * 2; strides[2] = (cuuint64_t)2 * H * W * x_ld * 2;
      strides[3] = (cuuint64_t)D * H * W * x_ld * 2;
    } else {
      dims[0] = (cuuint64_t)cext; dims[1] = (cuuint64_t)W; dims[2] = (cuuint64_t)H; dims[3] = (cuuint64_t)D; dims[4] = (cuuint64_t)N;
      strides[0] = (cuuint64_t)x_ld * 2; strides[1] = (cuuint64_t)W * x_ld * 2; strides[2] = (cuuint64_t)H * W * x_ld * 2;
      strides[3] = (cuuint64_t)D * H * W * x_ld * 2;
    }
    cuuint32_t box[5] = {(cuuint32_t)p.KC, (cuuint32_t)(p.kwfuse ? p.tw + 2 : p.tw), (cuuint32_t)p.th, (cuuint32_t)p.td, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&map_x, tdt, 5, const_cast<void*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { seg3d_set_error("conv_tc: cuTensorMapEncodeTiled(x) failed with %d", (int)r); return SEG3D_ECUDA; }
  }
  {
    const int wk = p.split ? 2 * Cin : Cin;              // weight rows hold [whi | wlo] in the split mode
    cuuint64_t dims[2] = {(cuuint64_t)wk, (cuuint64_t)(p.conv == 1 ? 8 * Cout : (p.conv == 2 ? 8 * p.cout_real : 27 * Cout))};
    cuuint64_t strides[1] = {(cuuint64_t)wk * 2};
    cuuint32_t box[2] = {(cuuint32_t)p.KC, (cuuint32_t)Cout};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(&map_w, tdt, 2, const_cast<void*>(w), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { seg3d_set_error("conv_tc: cuTensorMapEncodeTiled(w) failed with %d", (int)r); return SEG3D_ECUDA; }
  }
  const size_t smem = 1024 + (size_t)stages * stage_bytes + (2 * stages + 4) * 8 + 64 + 256 * 4;
  const long long max_grid = (long long)ctas_per_sm * seg3d_num_sms();
  dim3 grid((unsigned)(ntiles < max_grid ? ntiles : max_grid));
  cudaError_t e = dtype == SEG3D_BF16 ? launch_tc<__nv_bfloat16>(grid, smem, st, map_x, map_w, p, bias, y, stats)
                                      : launch_tc<__half>(grid, smem, st, map_x, map_w, p, bias, y, stats);
  if (e != cudaSuccess) { seg3d_set_error("conv_tc kernel launch failed: %s", cudaGetErrorString(e)); return SEG3D_ECUDA; }
  return SEG3D_OK;
}

// dW (fp32 [27][Cin][Cout], accumulated) for the k3 convolution on the tensor cores; returns SEG3D_EUNSUPPORTED
// for shapes it does not take so the caller can use the SIMT kernel.
int seg3d_wgrad_tc(int dtype, const void* x, int x_ld, int Cin, const void* dy, int dy_ld, int Cout, float* dw,
                   int N, int D, int H, int W, cudaStream_t st) {
  if (dtype != SEG3D_F16 && dtype != SEG3D_BF16) return SEG3D_EUNSUPPORTED;
  if (Cin % 16 || Cout % 16 || x_ld % 8 || dy_ld % 8) return SEG3D_EUNSUPPORTED;
  if (env_int("SEG3D_TC_WGRAD", 1) == 0) return SEG3D_EUNSUPPORTED;
  EncodeTiledFn encode = get_encode();
  if (!encode) return SEG3D_EUNSUPPORTED;
  WgParams p;
  memset(&p, 0, sizeof(p));
  p.Cin = Cin; p.Cout = Cout; p.D = D; p.H = H; p.W = W; p.N = N;
  p.nblk = Cin >= 64 ? 64 : Cin;                    // 16, 32 or 64 (Cin = 48 etc. not produced by the networks)
  if (Cin % p.nblk || (p.nblk != 16 && p.nblk != 32 && p.nblk != 64)) return SEG3D_EUNSUPPORTED;
  p.mblk = Cout >= 128 ? 128 : Cout;
  if (Cout % p.mblk) return SEG3D_EUNSUPPORTED;
  p.n_ci_blk = Cin / p.nblk; p.n_co_blk = Cout / p.mblk;
  p.taps_per_group = p.nblk <= 32 ? 9 : 3;
  p.ngroups = 27 / p.taps_per_group;
  p.ntx = (W + 7) / 8; p.nty = (H + 15) / 16;
  const long long ntiles = (long long)p.ntx * p.nty * D * N;
  if (ntiles <= 0 || ntiles >= (1ll << 31)) return SEG3D_EUNSUPPORTED;
  p.ntiles = (int)ntiles;
  p.a_atoms = (p.mblk + 63) / 64;
  // M = 128 always reads two 64-channel atoms (LBO = 16 KB apart); with one real atom the second read lands in the
  // next slab of the ring (valid shared memory, values ignored: they only reach accumulator rows >= 64)
  p.a_bytes = p.a_atoms * 16384;
  p.a_tx = p.a_atoms * 16384;
  p.b_row_bytes = p.nblk * 2;
  p.b_tx = 180 * p.b_row_bytes;
  p.b_bytes = (p.b_tx + 1023) & ~1023;
  p.stages = (200 * 1024) / (p.a_bytes + p.b_bytes); if (p.stages > 8) p.stages = 8;
  p.a_sbo = 1024; p.a_lbo = 16384; p.a_layout = 2;
  p.b_sbo = 10 * p.b_row_bytes;
  p.b_layout = p.b_row_bytes == 128 ? 2u : (p.b_row_bytes == 64 ? 4u : 6u);
  const int cols = p.taps_per_group * p.nblk;
  p.tmem_cols = cols <= 32 ? 32 : (cols <= 64 ? 64 : (cols <= 128 ? 128 : (cols <= 256 ? 256 : 512)));
  const uint32_t fmt = dtype == SEG3D_BF16 ? 1u : 0u;
  // MN-major A and B (bits 15, 16), M = 128, N = ci block
  p.idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(p.nblk >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  p.idesc3 = (1u << 4) | (fmt << 7) | (fmt << 10) | (1u << 15) | (1u << 16) | ((uint32_t)((3 * p.nblk) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  p.merge_kw = env_int("SEG3D_WGRAD_MERGE_KW", 1);
  const CUtensorMapDataType tdt = dtype == SEG3D_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUtensorMap map_dy, map_x;
  {
    cuuint64_t dims[5] = {(cuuint64_t)Cout, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)N};
    cuuint64_t strides[4] = {(cuuint64_t)dy_ld * 2, (cuuint64_t)W * dy_ld * 2, (cuuint64_t)H * W * dy_ld * 2, (cuuint64_t)D * H * W * dy_ld * 2};
    cuuint32_t box[5] = {64, 8, 16, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&map_dy, tdt, 5, const_cast<void*>(dy), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { seg3d_set_error("wgrad_tc: cuTensorMapEncodeTiled(dy) failed with %d", (int)r); return SEG3D_ECUDA; }
  }
  {
    const CUtensorMapSwizzle sw = p.b_row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (p.b_row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
    cuuint64_t dims[5] = {(cuuint64_t)Cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)N};
    cuuint64_t strides[4] = {(cuuint64_t)x_ld * 2, (cuuint64_t)W * x_ld * 2, (cuuint64_t)H * W * x_ld * 2, (cuuint64_t)D * H * W * x_ld * 2};
    cuuint32_t box[5] = {(cuuint32_t)p.nblk, 10, 18, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&map_x, tdt, 5, const_cast<void*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { seg3d_set_error("wgrad_tc: cuTensorMapEncodeTiled(x) failed with %d", (int)r); return SEG3D_ECUDA; }
  }
  const int combos = p.n_co_blk * p.n_ci_blk * p.ngroups;
  const int ctas_per_sm = (512 / p.tmem_cols) < 1 ? 1 : ((512 / p.tmem_cols) > 1 ? 1 : 1);   // smem ring ~170 KB: one CTA per SM
  // one CTA per SM and one wave: rounding the K split UP (e.g. 3 x 50 = 150 CTAs on 148 SMs) leaves two CTAs for a
  // second wave that doubles the run time
  long long ksplit = ((long long)ctas_per_sm * seg3d_num_sms()) / combos;
  if (ksplit < 1) ksplit = 1;
  if (ksplit > ntiles) ksplit = ntiles;
  const size_t smem = 1024 + (size_t)p.stages * (p.a_bytes + p.b_bytes) + 16384 + (2 * p.stages + 1) * 8 + 64;
  dim3 grid((unsigned)ksplit, (unsigned)combos);
  cudaError_t e = cudaSuccess;
#define SEG3D_LAUNCH_WG(TT, NB, TP)                                                                                          \
  { e = cudaFuncSetAttribute(conv3d_k3_wgrad_tc_kernel<TT, NB, TP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
    if (e == cudaSuccess) { conv3d_k3_wgrad_tc_kernel<TT, NB, TP><<<grid, TC_THREADS, smem, st>>>(map_dy, map_x, p, dw); e = cudaGetLastError(); } }
  if (dtype == SEG3D_BF16) {
    if (p.nblk == 64) SEG3D_LAUNCH_WG(__nv_bfloat16, 64, 3) else if (p.nblk == 32) SEG3D_LAUNCH_WG(__nv_bfloat16, 32, 9) else SEG3D_LAUNCH_WG(__nv_bfloat16, 16, 9)
  } else {
    if (p.nblk == 64) SEG3D_LAUNCH_WG(__half, 64, 3) else if (p.nblk == 32) SEG3D_LAUNCH_WG(__half, 32, 9) else SEG3D_LAUNCH_WG(__half, 16, 9)
  }
#undef SEG3D_LAUNCH_WG
  if (e != cudaSuccess) { seg3d_set_error("conv3d_k3_wgrad_tc_kernel launch failed: %s", cudaGetErrorString(e)); return SEG3D_ECUDA; }
  return SEG3D_OK;
}

// Tensor-core wgrad of the stride-2 convolutions.  mode: SEG3D_CONV_K2S2 (x dims D,H,W; dy = D/2..) or
// SEG3D_CONV_T2S2 (x dims D,H,W; dy = 2D..).  dw in the SIMT layouts of seg3d_conv3d_fwd.
int seg3d_wgrad_s2_tc(int mode, int dtype, const void* x, int x_ld, int Cin, const void* dy, int dy_ld, int Cout, float* dw,
                      int N, int D, int H, int W, cudaStream_t st) {
  if (dtype != SEG3D_F16 && dtype != SEG3D_BF16) return SEG3D_EUNSUPPORTED;
  if (Cin % 16 || Cout % 16 || x_ld % 8 || dy_ld % 8) return SEG3D_EUNSUPPORTED;
  if (env_int("SEG3D_TC_WGRAD", 1) == 0) return SEG3D_EUNSUPPORTED;
  if (mode == SEG3D_CONV_K2S2 && (D % 2 || H % 2 || W % 2)) return SEG3D_EUNSUPPORTED;
  EncodeTiledFn encode = get_encode();
  if (!encode) return SEG3D_EUNSUPPORTED;
  Wg2Params p;
  memset(&p, 0, sizeof(p));
  p.mode = mode == SEG3D_CONV_K2S2 ? 1 : 2;
  p.Cin = Cin; p.Cout = Cout; p.N = N;
  p.nblk = Cin >= 64 ? 64 : Cin;
  if (Cin % p.nblk || (p.nblk != 16 && p.nblk != 32 && p.nblk != 64)) return SEG3D_EUNSUPPORTED;
  p.mblk = Cout >= 128 ? 128 : Cout;
  if (Cout % p.mblk) return SEG3D_EUNSUPPORTED;
  p.n_ci_blk = Cin / p.nblk; p.n_co_blk = Cout / p.mblk;
  // low-resolution iteration grid
  const int Dl = p.mode == 1 ? D / 2 : D, Hl = p.mode == 1 ? H / 2 : H, Wl = p.mode == 1 ? W / 2 : W;
  p.D = Dl; p.H = Hl; p.W = Wl;
  p.ntx = (Wl + 7) / 8; p.nty = (Hl + 15) / 16;
  const long long ntiles = (long long)p.ntx * p.nty * Dl * N;
  if (ntiles <= 0 || ntiles >= (1ll << 31)) return SEG3D_EUNSUPPORTED;
  p.ntiles = (int)ntiles;
  p.a_atoms = (p.mblk + 63) / 64;
  p.a_slab = p.a_atoms * 16384;
  p.b_row_bytes = p.nblk * 2;
  p.b_slab = (128 * p.b_row_bytes + 1023) & ~1023;
  p.a_bytes = p.mode == 1 ? p.a_slab : 2 * p.a_slab;
  p.b_bytes = p.mode == 1 ? 2 * p.b_slab : p.b_slab;
  p.tx_bytes = (p.mode == 1 ? 1 : 2) * p.a_atoms * 16384 + (p.mode == 1 ? 2 : 1) * 128 * p.b_row_bytes;
  p.stages = (190 * 1024) / (p.a_bytes + p.b_bytes); if (p.stages > 8) p.stages = 8;
  if (p.stages < 2) return SEG3D_EUNSUPPORTED;
  p.b_sbo = 8 * p.b_row_bytes;
  p.b_layout = p.b_row_bytes == 128 ? 2u : (p.b_row_bytes == 64 ? 4u : 6u);
  const int cols = 2 * p.nblk;
  p.tmem_cols = cols <= 32 ? 32 : (cols <= 64 ? 64 : 128);
  const uint32_t fmt = dtype == SEG3D_BF16 ? 1u : 0u;
  p.idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(p.nblk >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  const CUtensorMapDataType tdt = dtype == SEG3D_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const CUtensorMapSwizzle swb = p.b_row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (p.b_row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  CUtensorMap map_dy, map_x;
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  // dense low-resolution tensor and folded high-resolution tensor
  const void* lo_ptr = p.mode == 1 ? dy : x;   const int lo_ld = p.mode == 1 ? dy_ld : x_ld;   const int lo_C = p.mode == 1 ? Cout : Cin;
  const void* hi_ptr = p.mode == 1 ? x : dy;   const int hi_ld = p.mode == 1 ? x_ld : dy_ld;   const int hi_C = p.mode == 1 ? Cin : Cout;
  const int Wh = 2 * Wl, Hh = 2 * Hl, Dh = 2 * Dl;
  p.fold_ld = hi_ld; p.foldW = Wl; p.foldH = Hl;
  CUtensorMap map_lo, map_hi;
  {
    cuuint64_t dims[5] = {(cuuint64_t)lo_C, (cuuint64_t)Wl, (cuuint64_t)Hl, (cuuint64_t)Dl, (cuuint64_t)N};
    cuuint64_t strides[4] = {(cuuint64_t)lo_ld * 2, (cuuint64_t)Wl * lo_ld * 2, (cuuint64_t)Hl * Wl * lo_ld * 2, (cuuint64_t)Dl * Hl * Wl * lo_ld * 2};
    cuuint32_t box[5] = {(cuuint32_t)(p.mode == 1 ? 64 : p.nblk), 8, 16, 1, 1};
    CUresult r = encode(&map_lo, tdt, 5, const_cast<void*>(lo_ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        p.mode == 1 ? CU_TENSOR_MAP_SWIZZLE_128B : swb, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { seg3d_set_error("wgrad_s2_tc: cuTensorMapEncodeTiled(lo) failed with %d", (int)r); return SEG3D_ECUDA; }
  }
  {
    cuuint64_t dims[5] = {(cuuint64_t)hi_ld + hi_C, (cuuint64_t)Wh, (cuuint64_t)Hh, (cuuint64_t)Dh / 2, (cuuint64_t)N};
    cuuint64_t strides[4] = {(cuuint64_t)2 * hi_ld * 2, (cuuint64_t)2 * Wh * hi_ld * 2, (cuuint64_t)2 * Hh * Wh * hi_ld * 2, (cuuint64_t)Dh * Hh * Wh * hi_ld * 2};
    cuuint32_t box[5] = {(cuuint32_t)(p.mode == 1 ? p.nblk : 64), 8, 16, 1, 1};
    CUresult r = encode(&map_hi, tdt, 5, const_cast<void*>(hi_ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        p.mode == 1 ? swb : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { seg3d_set_error("wgrad_s2_tc: cuTensorMapEncodeTiled(hi) failed with %d", (int)r); return SEG3D_ECUDA; }
  }
  if (p.mode == 1) { map_dy = map_lo; map_x = map_hi; } else { map_dy = map_hi; map_x = map_lo; }
  const int combos = p.n_co_blk * p.n_ci_blk * 4;
  long long ksplit = (long long)seg3d_num_sms() / combos;        // one wave of one CTA per SM (see seg3d_wgrad_tc)
  if (ksplit < 1) ksplit = 1;
  if (ksplit > ntiles) ksplit = ntiles;
  const size_t smem = 1024 + (size_t)p.stages * (p.a_bytes + p.b_bytes) + 16384 + (2 * p.stages + 1) * 8 + 64;
  dim3 grid((unsigned)ksplit, (unsigned)combos);
  cudaError_t e = cudaSuccess;
#define SEG3D_LAUNCH_WG2(TT, NB, MD)                                                                                         \
  { e = cudaFuncSetAttribute(conv3d_s2_wgrad_tc_kernel<TT, NB, MD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  \
    if (e == cudaSuccess) { conv3d_s2_wgrad_tc_kernel<TT, NB, MD><<<grid, TC_THREADS, smem, st>>>(map_dy, map_x, p, dw); e = cudaGetLastError(); } }
#define SEG3D_LAUNCH_WG2_T(TT)                                                                                               \
  if (p.mode == 1) { if (p.nblk == 64) SEG3D_LAUNCH_WG2(TT, 64, 1) else if (p.nblk == 32) SEG3D_LAUNCH_WG2(TT, 32, 1) else SEG3D_LAUNCH_WG2(TT, 16, 1) } \
  else             { if (p.nblk == 64) SEG3D_LAUNCH_WG2(TT, 64, 2) else if (p.nblk == 32) SEG3D_LAUNCH_WG2(TT, 32, 2) else SEG3D_LAUNCH_WG2(TT, 16, 2) }
  if (dtype == SEG3D_BF16) { SEG3D_LAUNCH_WG2_T(__nv_bfloat16) } else { SEG3D_LAUNCH_WG2_T(__half) }
#undef SEG3D_LAUNCH_WG2_T
#undef SEG3D_LAUNCH_WG2
  if (e != cudaSuccess) { seg3d_set_error("conv3d_s2_wgrad_tc_kernel launch failed: %s", cudaGetErrorString(e)); return SEG3D_ECUDA; }
  return SEG3D_OK;
}
