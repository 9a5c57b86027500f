// Tensor-core TRAINING trunk of the generator: forward, data-gradient and weight-gradient of the
// residual-dense-block 3x3 convolutions (srgan_train.py:292-358, 467-486; autograd of the same links in
// g_loss.backward(), :1256) as tcgen05 implicit GEMMs on a "flat-padded" activation layout.
//
// Layout ("flat slab"): every image is stored WITH its one-pixel zero border, and the padded images
// are flattened into one position axis:  p = (img * (H+2) + y) * (W+2) + x,  P = N (H+2)(W+2).
//   bf16 slab8 : [C/8][Pg][8]     fp32 slab4 : [C/4][Pg][4]     Pg = G0 + 128*ceil(P/128) + G0
// (G0 = zero guard >= W+3). Border and guard positions are zero and are never written, so a 3x3 'same'
// convolution is nine SHIFTED GEMMs over the position axis: out[p] = sum_tap W_tap . in[p + (ky-1)(W+2) + kx-1].
// An M=128 UMMA tile is 128 consecutive positions (no spatial tile quantisation: the 9x9 training tiles
// of the reference keep 81/121 = 67 % of the MMA rows useful, a 16x16 spatial tile would keep 32 %).
//   * forward / dgrad : A = positions x channels (K-major core matrices: 8 positions x 8 channels =
//     128 contiguous bytes straight from HBM by one 1-D bulk copy per slab), tap = +16 B * shift on the
//     descriptor start address; B = pre-packed filters (dgrad: transposed + flipped).
//   * wgrad : dW[o][c][tap] = sum_p g[o][p] a[c][p + shift]: the SAME buffers are MN-major operands
//     (K = position, 16-byte pitch), again with the tap as a start-address shift; split over position
//     ranges, partial sums reduced by a second kernel.
// Epilogues are table driven per 32 output columns (bias, residual adds, LeakyReLU or its derivative
// mask, fp32 and/or bf16 stores), so one kernel covers every layer of the forward and backward chains.
#include "flat_records.cuh"

namespace dbm {

static int g_flat_swap_wgrad = 0;  // debug: swap LBO/SBO of the MN-major descriptors

struct FlatGeom {
  int n, H, W, Hp, Wp, img, P, tiles, G0, Pg, halo, R;
  int oh, ow;  // output window written by the conv epilogue: rows 1..oh, columns 1..ow (<= H, W)
};

static FlatGeom flat_geom(int n, int h, int w) {
  FlatGeom g;
  g.n = n; g.H = h; g.W = w; g.Hp = h + 2; g.Wp = w + 2; g.img = g.Hp * g.Wp;
  g.P = n * g.img;
  g.tiles = (g.P + 127) / 128;
  g.halo = g.Wp + 1;
  g.G0 = (g.halo + 7) & ~7;
  g.Pg = g.G0 + g.tiles * 128 + g.G0;
  g.R = 128 + 2 * g.halo;
  g.oh = h; g.ow = w;
  return g;
}

constexpr int kFlatThreads = 192;  // warp0 bulk-copy producer, warp1 MMA issuer, warps2-5 epilogue
constexpr int kFlatSmem = 208 * 1024;
constexpr int kFlatMaxStages = 8;

__device__ __forceinline__ uint32_t idesc_bf16_rt(uint32_t M, uint32_t N, uint32_t mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (mn_major << 15) | (mn_major << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// One 32-column block of an accumulator row -> table-driven epilogue (bias, residual adds, LeakyReLU or its
// derivative mask, fp32 / bf16 stores) at flat position ``pos``.
__device__ __forceinline__ void flat_epi_apply(const FlatEpiBlock& e, const uint32_t (&acc)[32], long ych, long yf,
                                               long pos, const FlatGeom& g) {
  float v[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(acc[i]);
  if (e.bias) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __fadd_rn(v[i], __ldg(e.bias + ych + i));
  }
  if (e.add1) {
    const float s1 = e.s1, be = e.beta;
#pragma unroll
    for (int s4 = 0; s4 < 8; ++s4) {
      const float4 rr = *reinterpret_cast<const float4*>(e.add1 + yf + ((long)s4 * g.Pg + pos) * 4);
      // explicit fused form (one rounding when s1 == 1): the image-resident kernel (umma_local.cu) computes the
      // same expression and is checked bit for bit against this one
      v[4 * s4 + 0] = __fmaf_rn(be, v[4 * s4 + 0], s1 * rr.x);
      v[4 * s4 + 1] = __fmaf_rn(be, v[4 * s4 + 1], s1 * rr.y);
      v[4 * s4 + 2] = __fmaf_rn(be, v[4 * s4 + 2], s1 * rr.z);
      v[4 * s4 + 3] = __fmaf_rn(be, v[4 * s4 + 3], s1 * rr.w);
    }
  }
  if (e.add2) {
    const float be = e.beta2;
#pragma unroll
    for (int s4 = 0; s4 < 8; ++s4) {
      const float4 rr = *reinterpret_cast<const float4*>(e.add2 + yf + ((long)s4 * g.Pg + pos) * 4);
      v[4 * s4 + 0] = __fmaf_rn(be, v[4 * s4 + 0], rr.x);
      v[4 * s4 + 1] = __fmaf_rn(be, v[4 * s4 + 1], rr.y);
      v[4 * s4 + 2] = __fmaf_rn(be, v[4 * s4 + 2], rr.z);
      v[4 * s4 + 3] = __fmaf_rn(be, v[4 * s4 + 3], rr.w);
    }
  }
  if (e.act) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = lrelu(v[i]);
  }
  if (e.mask) {
#pragma unroll
    for (int s8 = 0; s8 < 4; ++s8) {
      const uint4 mm = *reinterpret_cast<const uint4*>(e.mask + yf + ((long)s8 * g.Pg + pos) * 8);
      const uint32_t w4[4] = {mm.x, mm.y, mm.z, mm.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        // bf16 sign bits: low half = even channel, high half = odd channel
        if (w4[j] & 0x00008000u) v[8 * s8 + 2 * j] *= kLreluSlope;
        if (w4[j] & 0x80000000u) v[8 * s8 + 2 * j + 1] *= kLreluSlope;
      }
    }
  }
  if (e.out_f32) {
#pragma unroll
    for (int s4 = 0; s4 < 8; ++s4)
      *reinterpret_cast<float4*>(e.out_f32 + yf + ((long)s4 * g.Pg + pos) * 4) =
          make_float4(v[4 * s4], v[4 * s4 + 1], v[4 * s4 + 2], v[4 * s4 + 3]);
  }
  if (e.out_bf16) {
    const float sc = e.out_scale;
#pragma unroll
    for (int s8 = 0; s8 < 4; ++s8) {
      uint4 o;
      __nv_bfloat162 t0 = __floats2bfloat162_rn(sc * v[8 * s8 + 0], sc * v[8 * s8 + 1]);
      __nv_bfloat162 t1 = __floats2bfloat162_rn(sc * v[8 * s8 + 2], sc * v[8 * s8 + 3]);
      __nv_bfloat162 t2 = __floats2bfloat162_rn(sc * v[8 * s8 + 4], sc * v[8 * s8 + 5]);
      __nv_bfloat162 t3 = __floats2bfloat162_rn(sc * v[8 * s8 + 6], sc * v[8 * s8 + 7]);
      o.x = *reinterpret_cast<uint32_t*>(&t0);
      o.y = *reinterpret_cast<uint32_t*>(&t1);
      o.z = *reinterpret_cast<uint32_t*>(&t2);
      o.w = *reinterpret_cast<uint32_t*>(&t3);
      *reinterpret_cast<uint4*>(e.out_bf16 + yf + ((long)s8 * g.Pg + pos) * 8) = o;
    }
  }
}

__global__ void __launch_bounds__(kFlatThreads, 1)
flat_conv_kernel(const __grid_constant__ FlatLaunch L, const FlatGeom g) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)smem;
  uint64_t* empty = full + kFlatMaxStages;
  uint64_t* tfull = empty + kFlatMaxStages;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = (uint32_t*)(tempty + 2);
  uint8_t* stages = smem + 1024;

  const int N = L.nout;
  const uint32_t slab_bytes = (uint32_t)g.R * 16u;
  const uint32_t a_bytes = 2u * slab_bytes, b_bytes = 288u * (uint32_t)N, stage_bytes = a_bytes + b_bytes;
  int nst = (kFlatSmem - 2048) / (int)stage_bytes;
  if (nst > kFlatMaxStages) nst = kFlatMaxStages;
  const int num_kc = L.cin / 16;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < nst; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 4); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < g.tiles; tile += gridDim.x) {
        const long pos0 = (long)g.G0 + (long)tile * 128 - g.halo;
        for (int kc = 0; kc < num_kc; ++kc) {
          mbar_wait(&empty[s], ph ^ 1);
          mbar_arrive_expect_tx(&full[s], stage_bytes);
          uint8_t* st = stages + (size_t)s * stage_bytes;
          bulk_load(st, L.in + ((long)(2 * kc) * g.Pg + pos0) * 8, slab_bytes, &full[s]);
          bulk_load(st + slab_bytes, L.in + ((long)(2 * kc + 1) * g.Pg + pos0) * 8, slab_bytes, &full[s]);
          bulk_load(st + a_bytes, L.wpacked + (size_t)blockIdx.y * L.w_chunk_stride + (size_t)kc * (b_bytes / 2),
                    b_bytes, &full[s]);
          if (++s == nst) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = idesc_bf16_rt(128, (uint32_t)N, 0);
    const uint32_t a_hi = desc_hi(128), b_hi = desc_hi(128);
    const uint32_t b_lbo = (uint32_t)(N / 8) * 128u;
    const uint32_t b_tap = (2u * b_lbo) >> 4;  // per-tap stride of the packed filters, 16-byte units
    const uint32_t st_u = smem_u32(stages);
    int s = 0, it = 0; uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < g.tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      mbar_wait(&tempty[buf], ((it >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d0 = tmem_base + (uint32_t)(buf * 256);
      for (int kc = 0; kc < num_kc; ++kc) {
        mbar_wait(&full[s], ph);
        tc_fence_after();
        const uint32_t a_lo = desc_lo(st_u + s * stage_bytes, slab_bytes);
        const uint32_t b_lo = desc_lo(st_u + s * stage_bytes + a_bytes, b_lbo);
        if (elect_one_sync()) {
#pragma unroll 1
          for (uint32_t tap = 0; tap < 9; ++tap) {
            const uint32_t a_off = (tap / 3) * (uint32_t)g.Wp + (tap % 3);   // ky * Wp + kx rows of 16 bytes
            umma_bf16(d0, make_desc(a_lo + a_off, a_hi), make_desc(b_lo + tap * b_tap, b_hi), idesc,
                      (kc | (int)tap) != 0 ? 1u : 0u);
          }
          umma_commit(&empty[s]);
          if (kc == num_kc - 1) umma_commit(&tfull[buf]);
        }
        __syncwarp();
        if (++s == nst) { s = 0; ph ^= 1; }
      }
    }
  } else {
    const int q = warp & 3;
    const int m = 32 * q + lane;
    int it = 0;
    for (int tile = blockIdx.x; tile < g.tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      mbar_wait(&tfull[buf], (it >> 1) & 1);
      tc_fence_after();
      const int p = tile * 128 + m;
      const int r = p % g.img;
      const int y = r / g.Wp, x = r - y * g.Wp;
      const bool interior = (p < g.P) && y >= 1 && y <= g.oh && x >= 1 && x <= g.ow;
      const long pos = (long)g.G0 + p;
      const int nblk = N / 32;
      const long ych = (long)blockIdx.y * N;        // first output channel of this chunk
      const long yf = ych * g.Pg;                   // slab-pointer advance in elements (fp32: x1 floats, bf16: x1 halves)
#pragma unroll 1
      for (int b = 0; b < nblk; ++b) {
        uint32_t acc[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(buf * 256 + b * 32), acc);
        tmem_wait_ld();
        if (interior) {
          const FlatEpiBlock& e = L.blk[b];
          flat_epi_apply(e, acc, ych, yf, pos, g);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[buf]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------
// Persistent chain: the same convolution pipeline over a DEVICE table of launches executed in order by one
// grid (one CTA per SM, tile -> CTA mapping fixed), so a 182-layer forward or data-gradient chain is one
// launch. Layer l may read what layers < l wrote within +-halo (< 128) positions of its tile: tile t of layer
// l waits for tiles t-1, t, t+1 of layer l-1 (flag = 4 epilogue warps; transitively every earlier layer is then
// complete on t-2..t+2, which also covers buffer re-use). Release/acquire as in umma_trunk.cu:
// st.global -> __syncwarp -> lane-0 __threadfence -> atomicAdd / ld.acquire.gpu -> fence.proxy.async -> bulk copy.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned int flat_ld_acquire(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__global__ void __launch_bounds__(kFlatThreads, 1)
flat_chain_kernel(const FlatLaunch* __restrict__ table, int count, const FlatGeom g, unsigned int* __restrict__ done,
                  uint32_t stage_bytes, int nst) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)smem;
  uint64_t* empty = full + kFlatMaxStages;
  uint64_t* tfull = empty + kFlatMaxStages;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = (uint32_t*)(tempty + 2);
  uint8_t* stages = smem + 1024;

  const uint32_t slab_bytes = (uint32_t)g.R * 16u;
  const uint32_t a_bytes = 2u * slab_bytes;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < nst; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 4); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ---- dependency wait + bulk-copy producer (converged warp; lanes 0..2 watch the three neighbour tiles) ----
    int s = 0; uint32_t ph = 0;
    for (int l = 0; l < count; ++l) {
      const __nv_bfloat16* in = table[l].in;
      const __nv_bfloat16* wp = table[l].wpacked;
      const int num_kc = table[l].cin / 16;
      const uint32_t b_bytes = 288u * (uint32_t)table[l].nout;
      for (int tile = blockIdx.x; tile < g.tiles; tile += gridDim.x) {
        if (l > 0) {
          const int nt = tile + lane - 1;
          if (lane < 3 && nt >= 0 && nt < g.tiles) {
            const unsigned int* f = done + (size_t)(l - 1) * g.tiles + nt;
            SpinGuard guard;
            while (flat_ld_acquire(f) < 4u) {
              if (guard.expired()) {
                printf("dbm: flat chain dependency timeout layer %d tile %d\n", l, tile);
                __trap();
              }
              __nanosleep(32);
            }
          }
          __syncwarp();
        }
        const long pos0 = (long)g.G0 + (long)tile * 128 - g.halo;
        for (int kc = 0; kc < num_kc; ++kc) {
          mbar_wait(&empty[s], ph ^ 1);
          if (lane == 0) {
            // order the acquired flags (generic proxy) before the bulk-copy reads (async proxy)
            asm volatile("fence.proxy.async.global;" ::: "memory");
            mbar_arrive_expect_tx(&full[s], a_bytes + b_bytes);
            uint8_t* st = stages + (size_t)s * stage_bytes;
            bulk_load(st, in + ((long)(2 * kc) * g.Pg + pos0) * 8, slab_bytes, &full[s]);
            bulk_load(st + slab_bytes, in + ((long)(2 * kc + 1) * g.Pg + pos0) * 8, slab_bytes, &full[s]);
            bulk_load(st + a_bytes, wp + (size_t)kc * (b_bytes / 2), b_bytes, &full[s]);
          }
          __syncwarp();
          if (++s == nst) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t a_hi = desc_hi(128), b_hi = desc_hi(128);
    const uint32_t st_u = smem_u32(stages);
    int s = 0, it = 0; uint32_t ph = 0;
    for (int l = 0; l < count; ++l) {
      const int N = table[l].nout;
      const int num_kc = table[l].cin / 16;
      const uint32_t idesc = idesc_bf16_rt(128, (uint32_t)N, 0);
      const uint32_t b_lbo = (uint32_t)(N / 8) * 128u;
      const uint32_t b_tap = (2u * b_lbo) >> 4;
      for (int tile = blockIdx.x; tile < g.tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1;
        mbar_wait(&tempty[buf], ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d0 = tmem_base + (uint32_t)(buf * 256);
        for (int kc = 0; kc < num_kc; ++kc) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t a_lo = desc_lo(st_u + s * stage_bytes, slab_bytes);
          const uint32_t b_lo = desc_lo(st_u + s * stage_bytes + a_bytes, b_lbo);
          if (elect_one_sync()) {
#pragma unroll 1
            for (uint32_t tap = 0; tap < 9; ++tap) {
              const uint32_t a_off = (tap / 3) * (uint32_t)g.Wp + (tap % 3);
              umma_bf16(d0, make_desc(a_lo + a_off, a_hi), make_desc(b_lo + tap * b_tap, b_hi), idesc,
                        (kc | (int)tap) != 0 ? 1u : 0u);
            }
            umma_commit(&empty[s]);
            if (kc == num_kc - 1) umma_commit(&tfull[buf]);
          }
          __syncwarp();
          if (++s == nst) { s = 0; ph ^= 1; }
        }
      }
    }
  } else {
    const int q = warp & 3;
    const int m = 32 * q + lane;
    int it = 0;
    for (int l = 0; l < count; ++l) {
      const FlatLaunch& L = table[l];
      const int nblk = L.nout / 32;
      for (int tile = blockIdx.x; tile < g.tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1;
        mbar_wait(&tfull[buf], (it >> 1) & 1);
        tc_fence_after();
        const int p = tile * 128 + m;
        const int r = p % g.img;
        const int y = r / g.Wp, x = r - y * g.Wp;
        const bool interior = (p < g.P) && y >= 1 && y <= g.oh && x >= 1 && x <= g.ow;
        const long pos = (long)g.G0 + p;
#pragma unroll 1
        for (int b = 0; b < nblk; ++b) {
          uint32_t acc[32];
          tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(buf * 256 + b * 32), acc);
          tmem_wait_ld();
          if (b == nblk - 1) {   // accumulator fully in registers: hand the TMEM buffer back before the stores
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[buf]);
          }
          if (interior) flat_epi_apply(L.blk[b], acc, 0, 0, pos, g);
        }
        // publish the tile: the warp's stores are ordered before lane 0's gpu-scope fence by __syncwarp
        __syncwarp();
        if (lane == 0) {
          __threadfence();
          atomicAdd(done + (size_t)l * g.tiles + tile, 1u);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------
// Weight gradient: dW[o][c][tap] = sum_p g[o][p] * a[c][p + shift(tap)]   (MN-major operands)
// ---------------------------------------------------------------------------------------------
constexpr int kWgradMaxStages = 6;

__global__ void __launch_bounds__(kFlatThreads, 1)
flat_wgrad_kernel(const WgradUnit* __restrict__ units, int num_units, const FlatGeom g, int swap) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)smem;
  uint64_t* empty = full + kWgradMaxStages;
  uint64_t* tfull = empty + kWgradMaxStages;
  uint64_t* tempty = tfull + 1;
  uint32_t* tmem_slot = (uint32_t*)(tempty + 1);
  uint8_t* stages = smem + 1024;

  const uint32_t slab_bytes = (uint32_t)g.R * 16u;
  const uint32_t a_bytes = 16u * slab_bytes, b_bytes = 4u * 2048u, stage_bytes = a_bytes + b_bytes;
  int nst = (kFlatSmem - 2048) / (int)stage_bytes;
  if (nst > kWgradMaxStages) nst = kWgradMaxStages;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < nst; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tfull, 1);
    mbar_init(tempty, 4);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
        const WgradUnit un = units[u];
        for (int blk = un.blk0; blk < un.blk0 + un.nblk; ++blk) {
          const long pos0 = (long)g.G0 + (long)blk * 128;
          mbar_wait(&empty[s], ph ^ 1);
          mbar_arrive_expect_tx(&full[s], (uint32_t)un.nslab * slab_bytes + b_bytes);
          uint8_t* st = stages + (size_t)s * stage_bytes;
          for (int sl = 0; sl < un.nslab; ++sl)
            bulk_load(st + sl * slab_bytes, un.act + ((long)sl * g.Pg + pos0 - g.halo) * 8, slab_bytes, &full[s]);
          for (int sl = 0; sl < 4; ++sl)
            bulk_load(st + a_bytes + sl * 2048, un.gout + ((long)sl * g.Pg + pos0) * 8, 2048, &full[s]);
          if (++s == nst) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = idesc_bf16_rt(128, 32, 1);
    // MN-major no-swizzle canonical layout ((8,m),(8,k)) : ((1,SBO),(16 B,LBO))  (cute mma_traits_sm100):
    // SBO = stride between 8-channel slabs, LBO = stride between groups of 8 positions (128 B)
    uint32_t a_lbo = 128, a_sbo = slab_bytes, b_lbo = 128, b_sbo = 2048;
    if (swap) { uint32_t t = a_lbo; a_lbo = a_sbo; a_sbo = t; t = b_lbo; b_lbo = b_sbo; b_sbo = t; }
    const uint32_t a_hi = desc_hi(a_sbo), b_hi = desc_hi(b_sbo);
    const uint32_t st_u = smem_u32(stages);
    int s = 0, it = 0; uint32_t ph = 0;
    for (int u = blockIdx.x; u < num_units; u += gridDim.x, ++it) {
      const int nblk = units[u].nblk;
      const uint32_t tapmask = units[u].tapmask ? (uint32_t)units[u].tapmask : 0x1FFu;
      mbar_wait(tempty, (it & 1) ^ 1);
      tc_fence_after();
      for (int b = 0; b < nblk; ++b) {
        mbar_wait(&full[s], ph);
        tc_fence_after();
        const uint32_t a_lo = desc_lo(st_u + s * stage_bytes, a_lbo);
        const uint32_t b_lo = desc_lo(st_u + s * stage_bytes + a_bytes, b_lbo);
        if (elect_one_sync()) {
#pragma unroll 1
          for (uint32_t tap = 0; tap < 9; ++tap) {
            if (!((tapmask >> tap) & 1u)) continue;
            const uint32_t a_tap = a_lo + (tap / 3) * (uint32_t)g.Wp + (tap % 3);
#pragma unroll 1
            for (uint32_t ks = 0; ks < 8; ++ks)
              umma_bf16(tmem_base + tap * 32, make_desc(a_tap + ks * 16, a_hi), make_desc(b_lo + ks * 16, b_hi), idesc,
                        (b | (int)ks) != 0 ? 1u : 0u);
          }
          umma_commit(&empty[s]);
          if (b == nblk - 1) umma_commit(tfull);
        }
        __syncwarp();
        if (++s == nst) { s = 0; ph ^= 1; }
      }
    }
  } else {
    const int q = warp & 3;
    const int c = 32 * q + lane;
    int it = 0;
    for (int u = blockIdx.x; u < num_units; u += gridDim.x, ++it) {
      const WgradUnit un = units[u];
      mbar_wait(tfull, it & 1);
      tc_fence_after();
#pragma unroll 1
      for (int tap = 0; tap < 9; ++tap) {
        if (un.tapmask && !((un.tapmask >> tap) & 1)) continue;
        uint32_t acc[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(tap * 32), acc);
        tmem_wait_ld();
        if (c < un.nslab * 8) {
#pragma unroll
          for (int o = 0; o < 32; ++o) un.partial[(tap * 32 + o) * 128 + c] = __uint_as_float(acc[o]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// grid = (entries, slices): blockIdx.y strides over the entry's 9 x 32 x nch outputs, so that an entry with many
// position splits (small layers: 4 entries x 74 splits) is still spread over every SM
__global__ void __launch_bounds__(256) flat_wgrad_reduce_kernel(const WgradReduce* __restrict__ table) {
  const WgradReduce e = table[blockIdx.x];
  const int total = 9 * 32 * e.nch;
  const int mode = e.mode & 0xFF;
  const int ovalid = ((e.mode >> 8) & 0xFF) ? ((e.mode >> 8) & 0xFF) : 32;
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < total; i += gridDim.y * blockDim.x) {
    const int c = i % e.nch;
    const int t = i / e.nch;
    const int o = t & 31, tap = t >> 5;
    if (o >= ovalid) continue;
    long dst;
    if (mode == 0) {
      dst = ((long)(e.o0 + o) * e.cin_total + e.c0 + c) * 9 + tap;
    } else {
      const int cg = e.c0 + c;
      const int ph = cg / e.cin_total, cc = cg - ph * e.cin_total;
      const int ky = 2 * (tap / 3 - 1) + (ph >> 1) + 1, kx = 2 * (tap % 3 - 1) + (ph & 1) + 1;
      if (ky < 0 || ky > 3 || kx < 0 || kx > 3) continue;   // structurally zero tap of the embedding
      dst = ((long)(e.o0 + o) * e.cin_total + cc) * 16 + ky * 4 + kx;
    }
    const float* src = e.partial + (tap * 32 + o) * 128 + c;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int k = 0;
    for (; k + 4 <= e.nsplit; k += 4) {   // four independent loads in flight per thread
      s0 += __ldg(src + (long)k * e.split_stride);
      s1 += __ldg(src + (long)(k + 1) * e.split_stride);
      s2 += __ldg(src + (long)(k + 2) * e.split_stride);
      s3 += __ldg(src + (long)(k + 3) * e.split_stride);
    }
    for (; k < e.nsplit; ++k) s0 += __ldg(src + (long)k * e.split_stride);
    e.dw[dst] += (s0 + s1) + (s2 + s3);
  }
}

struct BiasGradEntry {  // 16 bytes: db[0:32] += sum_p g[32 channels][p]
  const __nv_bfloat16* gout;
  float* db;
};

__global__ void flat_bias_grad_kernel(const BiasGradEntry* __restrict__ table, const FlatGeom g) {
  const BiasGradEntry e = table[blockIdx.x];
  __shared__ float red[8][32];
  const int sl = threadIdx.x & 3;             // slab (8 channels)
  const int lane_p = threadIdx.x >> 2;        // 64 position lanes
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const __nv_bfloat16* base = e.gout + ((long)sl * g.Pg + g.G0) * 8;
  for (int p = lane_p; p < g.P; p += 64) {
    const uint4 v = *reinterpret_cast<const uint4*>(base + (long)p * 8);
    const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      acc[2 * j] += __uint_as_float(w4[j] << 16);
      acc[2 * j + 1] += __uint_as_float(w4[j] & 0xFFFF0000u);
    }
  }
  // reduce over the 64 position lanes: lanes with equal (threadIdx.x & 3) within a warp, then across warps
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float a = acc[j];
    a += __shfl_xor_sync(0xFFFFFFFFu, a, 4);
    a += __shfl_xor_sync(0xFFFFFFFFu, a, 8);
    a += __shfl_xor_sync(0xFFFFFFFFu, a, 16);
    if ((threadIdx.x & 31) < 4) red[threadIdx.x >> 5][sl * 8 + j] = a;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
    e.db[threadIdx.x] += s;
  }
}

// ---- layout converters: NCHW fp32 <-> flat slabs (interior positions only) ---------------------
// mode 0: the (sh, sw) source image sits in the top-left corner of the (H, W) interior;
// mode 1: space-to-depth by 2: source pixel (y, x) of channel c -> channel ((y&1)*2 + (x&1)) * C + c at (y>>1, x>>1)
//         (a 4x4 stride-2 pad-1 convolution becomes a 3x3 stride-1 pad-1 one over the 4C phase channels).
__global__ void flat_from_nchw_kernel(const float* __restrict__ src, int C, int sh, int sw, int mode,
                                      __nv_bfloat16* dst8, float* dst4, float scale, const FlatGeom g) {
  const int c4n = (C + 3) / 4;
  const long total = (long)g.n * c4n * sh * sw;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    long t = i;
    const int x = t % sw; t /= sw;
    const int y = t % sh; t /= sh;
    const int n = t % g.n; t /= g.n;
    const int c4 = (int)t;
    int gy = y, gx = x, ch = c4 * 4;
    if (mode == 1) {
      ch += (((y & 1) << 1) | (x & 1)) * C;
      gy = y >> 1; gx = x >> 1;
    }
    const long pos = (long)g.G0 + ((long)n * g.Hp + gy + 1) * g.Wp + gx + 1;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
      v[j] = (c4 * 4 + j < C) ? scale * src[(((long)n * C + c4 * 4 + j) * sh + y) * sw + x] : 0.f;
    if (dst4) *reinterpret_cast<float4*>(dst4 + ((long)(ch >> 2) * g.Pg + pos) * 4) = make_float4(v[0], v[1], v[2], v[3]);
    if (dst8) {
      __nv_bfloat162 t0 = __floats2bfloat162_rn(v[0], v[1]);
      __nv_bfloat162 t1 = __floats2bfloat162_rn(v[2], v[3]);
      uint2 o;
      o.x = *reinterpret_cast<uint32_t*>(&t0);
      o.y = *reinterpret_cast<uint32_t*>(&t1);
      *reinterpret_cast<uint2*>(dst8 + ((long)(ch >> 3) * g.Pg + pos) * 8 + (ch & 4)) = o;
    }
  }
}

__global__ void flat_to_nchw_kernel(const float* __restrict__ src4, const __nv_bfloat16* __restrict__ src8,
                                    float* __restrict__ dst, int C, int dh, int dw, int mode, const FlatGeom g) {
  const long total = (long)g.n * C * dh * dw;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    long t = i;
    const int x = t % dw; t /= dw;
    const int y = t % dh; t /= dh;
    int c = t % C; t /= C;
    const int n = (int)t;
    int gy = y, gx = x;
    if (mode == 1) {
      c += (((y & 1) << 1) | (x & 1)) * C;
      gy = y >> 1; gx = x >> 1;
    }
    const long pos = (long)g.G0 + ((long)n * g.Hp + gy + 1) * g.Wp + gx + 1;
    dst[i] = src4 ? src4[((long)(c >> 2) * g.Pg + pos) * 4 + (c & 3)]
                  : __bfloat162float(src8[((long)(c >> 3) * g.Pg + pos) * 8 + (c & 7)]);
  }
}

// Vectorised forms for channel counts that are whole slabs: one thread moves a whole 16-byte slab element
// (4 fp32 / 8 bf16 channels of one position) -- the scalar kernels above use 4 of every 16 bytes they fetch.
template <int CG>   // 4: fp32 slab4 source, 8: bf16 slab8 source
__global__ void flat_to_nchw_vec_kernel(const void* __restrict__ src, float* __restrict__ dst, int C, int dh, int dw,
                                        int mode, const FlatGeom g) {
  const int cgn = C / CG;
  const long total = (long)g.n * cgn * dh * dw;
  const long plane = (long)dh * dw;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    long t = i;
    const int x = t % dw; t /= dw;
    const int y = t % dh; t /= dh;
    const int cg = t % cgn; t /= cgn;
    const int n = (int)t;
    int gy = y, gx = x, c = cg * CG;
    if (mode == 1) {
      c += (((y & 1) << 1) | (x & 1)) * C;
      gy = y >> 1; gx = x >> 1;
    }
    const long pos = (long)g.G0 + ((long)n * g.Hp + gy + 1) * g.Wp + gx + 1;
    float* d = dst + (((long)n * C + cg * CG) * dh + y) * dw + x;
    if (CG == 4) {
      const float4 v = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(src) + ((long)(c >> 2) * g.Pg + pos) * 4);
      d[0] = v.x; d[plane] = v.y; d[2 * plane] = v.z; d[3 * plane] = v.w;
    } else {
      const uint4 v = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(src) + ((long)(c >> 3) * g.Pg + pos) * 8);
      const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        d[(2 * j) * plane] = __uint_as_float(w4[j] << 16);
        d[(2 * j + 1) * plane] = __uint_as_float(w4[j] & 0xffff0000u);
      }
    }
  }
}

// bf16-only destination, C a multiple of 8: one thread gathers 8 channel planes and writes one 16-byte slab element
__global__ void flat_from_nchw_vec8_kernel(const float* __restrict__ src, int C, int sh, int sw, int mode,
                                           __nv_bfloat16* __restrict__ dst8, float scale, const FlatGeom g) {
  const int c8n = C / 8;
  const long total = (long)g.n * c8n * sh * sw;
  const long plane = (long)sh * sw;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    long t = i;
    const int x = t % sw; t /= sw;
    const int y = t % sh; t /= sh;
    const int c8 = t % c8n; t /= c8n;
    const int n = (int)t;
    int gy = y, gx = x, ch = c8 * 8;
    if (mode == 1) {
      ch += (((y & 1) << 1) | (x & 1)) * C;
      gy = y >> 1; gx = x >> 1;
    }
    const long pos = (long)g.G0 + ((long)n * g.Hp + gy + 1) * g.Wp + gx + 1;
    const float* sp = src + (((long)n * C + c8 * 8) * sh + y) * sw + x;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = scale * sp[j * plane];
    uint4 o;
    __nv_bfloat162 t0 = __floats2bfloat162_rn(v[0], v[1]);
    __nv_bfloat162 t1 = __floats2bfloat162_rn(v[2], v[3]);
    __nv_bfloat162 t2 = __floats2bfloat162_rn(v[4], v[5]);
    __nv_bfloat162 t3 = __floats2bfloat162_rn(v[6], v[7]);
    o.x = *reinterpret_cast<uint32_t*>(&t0);
    o.y = *reinterpret_cast<uint32_t*>(&t1);
    o.z = *reinterpret_cast<uint32_t*>(&t2);
    o.w = *reinterpret_cast<uint32_t*>(&t3);
    *reinterpret_cast<uint4*>(dst8 + ((long)(ch >> 3) * g.Pg + pos) * 8) = o;
  }
}

static int set_flat_attr() {
  if (int rc = ensure_dyn_smem((const void*)flat_conv_kernel, kFlatSmem)) return rc;
  if (int rc = ensure_dyn_smem((const void*)flat_wgrad_kernel, kFlatSmem)) return rc;
  return ensure_dyn_smem((const void*)flat_chain_kernel, kFlatSmem);
}

}  // namespace dbm

using namespace dbm;

static int g_flat_sm_reserve = 0;   // SMs the persistent weight-gradient kernel leaves to concurrent streams

extern "C" int dbm_flat_debug_set(int key, int value) {
  if (key == 1) g_flat_swap_wgrad = value;
  return DBM_OK;
}

extern "C" int dbm_set_sm_reserve(int n) {
  DBM_REQUIRE(n >= 0 && n < num_sms(), "set_sm_reserve: %d of %d SMs", n, num_sms());
  g_flat_sm_reserve = n;
  return DBM_OK;
}

extern "C" int dbm_flat_geometry(int n, int h, int w, int* out5_host) {
  DBM_REQUIRE(n > 0 && h > 0 && w > 0 && out5_host, "flat_geometry: bad arguments");
  const FlatGeom g = flat_geom(n, h, w);
  out5_host[0] = g.P; out5_host[1] = g.tiles; out5_host[2] = g.G0; out5_host[3] = g.Pg; out5_host[4] = g.R;
  return DBM_OK;
}

static int check_flat_shape(const FlatGeom& g, const char* who) {
  DBM_REQUIRE(g.n > 0 && g.H > 0 && g.W > 0, "%s: empty input", who);
  // widest stage: forward/dgrad N = 192 -> 2 R 16 + 288 * 192 bytes; wgrad -> 16 R 16 + 8192 bytes; need >= 2 stages
  DBM_REQUIRE(2 * (16 * g.R * 16 + 8192) <= kFlatSmem - 2048, "%s: image width %d too large for the flat trunk kernels "
              "(they serve the small training tiles; use the tiled inference kernels)", who, g.W);
  return DBM_OK;
}

extern "C" int dbm_flat_conv3x3_seq(const void* launches_host, int count, int n, int h, int w, int out_h, int out_w,
                                    cudaStream_t stream) {
  FlatGeom g = flat_geom(n, h, w);
  int rc = check_flat_shape(g, "flat_conv3x3");
  if (rc) return rc;
  rc = set_flat_attr();
  if (rc) return rc;
  DBM_REQUIRE(launches_host && count > 0, "flat_conv3x3: empty launch list");
  DBM_REQUIRE(out_h >= 0 && out_h <= h && out_w >= 0 && out_w <= w, "flat_conv3x3: output window %dx%d exceeds %dx%d",
              out_h, out_w, h, w);
  if (out_h > 0) g.oh = out_h;
  if (out_w > 0) g.ow = out_w;
  const FlatLaunch* L = (const FlatLaunch*)launches_host;
  for (int i = 0; i < count; ++i) {
    DBM_REQUIRE(L[i].cin % 16 == 0 && L[i].cin > 0, "flat_conv3x3[%d]: Cin=%d must be a multiple of 16", i, L[i].cin);
    DBM_REQUIRE(L[i].nout % 32 == 0 && L[i].nout >= 32 && L[i].nout <= 192,
                "flat_conv3x3[%d]: N=%d must be a multiple of 32 in [32, 192]", i, L[i].nout);
    DBM_REQUIRE(L[i].in && L[i].wpacked && (((uintptr_t)L[i].in | (uintptr_t)L[i].wpacked) & 15) == 0,
                "flat_conv3x3[%d]: null or unaligned operand", i);
    const int ny = L[i].ny > 0 ? L[i].ny : 1;
    DBM_REQUIRE(ny <= 64, "flat_conv3x3[%d]: %d output chunks", i, ny);
    int gx = num_sms() / ny;
    if (gx < 1) gx = 1;
    if (gx > g.tiles) gx = g.tiles;
    flat_conv_kernel<<<dim3(gx, ny), kFlatThreads, kFlatSmem, stream>>>(L[i], g);
  }
  return check_launch("flat_conv_kernel");
}

extern "C" int dbm_flat_conv3x3_chain(const void* launches_host, const void* launches_dev, int count, int n, int h,
                                      int w, int out_h, int out_w, void* flags_dev, cudaStream_t stream) {
  FlatGeom g = flat_geom(n, h, w);
  int rc = check_flat_shape(g, "flat_chain");
  if (rc) return rc;
  rc = set_flat_attr();
  if (rc) return rc;
  DBM_REQUIRE(launches_host && launches_dev && flags_dev && count > 0, "flat_chain: empty launch list");
  DBM_REQUIRE(out_h >= 0 && out_h <= h && out_w >= 0 && out_w <= w, "flat_chain: output window %dx%d exceeds %dx%d",
              out_h, out_w, h, w);
  DBM_REQUIRE(g.halo <= 128, "flat_chain: image width %d: the halo must stay within the neighbouring tile", w);
  if (out_h > 0) g.oh = out_h;
  if (out_w > 0) g.ow = out_w;
  const FlatLaunch* L = (const FlatLaunch*)launches_host;
  int nmax = 0;
  for (int i = 0; i < count; ++i) {
    DBM_REQUIRE(L[i].cin % 16 == 0 && L[i].cin > 0, "flat_chain[%d]: Cin=%d must be a multiple of 16", i, L[i].cin);
    DBM_REQUIRE(L[i].nout % 32 == 0 && L[i].nout >= 32 && L[i].nout <= 192,
                "flat_chain[%d]: N=%d must be a multiple of 32 in [32, 192]", i, L[i].nout);
    DBM_REQUIRE(L[i].in && L[i].wpacked && (((uintptr_t)L[i].in | (uintptr_t)L[i].wpacked) & 15) == 0,
                "flat_chain[%d]: null or unaligned operand", i);
    DBM_REQUIRE(L[i].ny <= 1, "flat_chain[%d]: output-channel chunks are not supported in a chain", i);
    if (L[i].nout > nmax) nmax = L[i].nout;
  }
  // one stage size for the whole chain (the widest layer's), so the ring layout never changes under in-flight stages
  const uint32_t stage_bytes = 2u * (uint32_t)g.R * 16u + 288u * (uint32_t)nmax;
  int nst = (kFlatSmem - 2048) / (int)stage_bytes;
  if (nst > kFlatMaxStages) nst = kFlatMaxStages;
  DBM_REQUIRE(nst >= 2, "flat_chain: stage of %u bytes does not fit twice", stage_bytes);
  // every CTA must be co-resident (tiles spin on flags set by other CTAs): bounded by the occupancy query
  int resident = 0;
  {
    int rc2 = resident_ctas((const void*)flat_chain_kernel, kFlatThreads, kFlatSmem, &resident);
    if (rc2) return rc2;
  }
  if (resident > num_sms()) resident = num_sms();
  const int grid = g.tiles < resident ? g.tiles : resident;
  DBM_CUDA(cudaMemsetAsync(flags_dev, 0, (size_t)count * g.tiles * sizeof(unsigned int), stream));
  flat_chain_kernel<<<grid, kFlatThreads, kFlatSmem, stream>>>((const FlatLaunch*)launches_dev, count, g,
                                                               (unsigned int*)flags_dev, stage_bytes, nst);
  return check_launch("flat_chain_kernel");
}

extern "C" int dbm_flat_wgrad_ctas(const void* units_dev, int num_units, int n, int h, int w, int max_ctas,
                                   cudaStream_t stream);
extern "C" int dbm_flat_wgrad(const void* units_dev, int num_units, int n, int h, int w, cudaStream_t stream) {
  return dbm_flat_wgrad_ctas(units_dev, num_units, n, h, w, 0, stream);
}

// max_ctas > 0: upper bound of the persistent grid for THIS launch (two weight-gradient kernels of different models
// running side by side each get a share of the SMs instead of the second one squeezing into what the first left free)
extern "C" int dbm_flat_wgrad_ctas(const void* units_dev, int num_units, int n, int h, int w, int max_ctas,
                                   cudaStream_t stream) {
  const FlatGeom g = flat_geom(n, h, w);
  int rc = check_flat_shape(g, "flat_wgrad");
  if (rc) return rc;
  rc = set_flat_attr();
  if (rc) return rc;
  DBM_REQUIRE(units_dev && num_units > 0, "flat_wgrad: empty unit table");
  // The training step runs the discriminator's ~150 small dependent kernels on a high-priority stream beside this
  // kernel; a persistent grid on every SM would stall that chain for the whole launch, so a few SMs can be left free
  // (dbm_set_sm_reserve(n): the units are dealt round-robin, results do not depend on the grid size)
  int cap = num_sms() - g_flat_sm_reserve;
  if (max_ctas > 0 && max_ctas < cap) cap = max_ctas;
  if (cap < 1) cap = 1;
  const int grid = num_units < cap ? num_units : cap;
  flat_wgrad_kernel<<<grid, kFlatThreads, kFlatSmem, stream>>>((const WgradUnit*)units_dev, num_units, g,
                                                                g_flat_swap_wgrad);
  return check_launch("flat_wgrad_kernel");
}

extern "C" int dbm_flat_wgrad_reduce(const void* entries_dev, int count, cudaStream_t stream) {
  DBM_REQUIRE(entries_dev && count > 0, "flat_wgrad_reduce: empty table");
  // >= 4 blocks per SM in total, at most one block per 256 outputs of the widest entry (9 x 32 x 128)
  int slices = ceil_div(4L * num_sms(), count);
  if (slices > 144) slices = 144;
  flat_wgrad_reduce_kernel<<<dim3(count, slices), 256, 0, stream>>>((const WgradReduce*)entries_dev);
  return check_launch("flat_wgrad_reduce_kernel");
}

extern "C" int dbm_flat_bias_grad(const void* entries_dev, int count, int n, int h, int w, cudaStream_t stream) {
  DBM_REQUIRE(entries_dev && count > 0, "flat_bias_grad: empty table");
  const FlatGeom g = flat_geom(n, h, w);
  flat_bias_grad_kernel<<<count, 256, 0, stream>>>((const BiasGradEntry*)entries_dev, g);
  return check_launch("flat_bias_grad_kernel");
}

extern "C" int dbm_flat_from_nchw_ex(const float* src, int c, int src_h, int src_w, int mode, void* dst_slab8,
                                     float* dst_slab4, float scale, int n, int h, int w, cudaStream_t stream) {
  DBM_REQUIRE(c > 0 && (mode == 0 || (mode == 1 && c % 8 == 0)), "flat_from_nchw: bad C=%d for mode %d", c, mode);
  DBM_REQUIRE(src && (dst_slab8 || dst_slab4), "flat_from_nchw: null pointer");
  if (mode == 0) DBM_REQUIRE(src_h <= h && src_w <= w, "flat_from_nchw: %dx%d source exceeds the %dx%d interior", src_h, src_w, h, w);
  else DBM_REQUIRE((src_h + 1) / 2 <= h && (src_w + 1) / 2 <= w, "flat_from_nchw: space-to-depth of %dx%d exceeds %dx%d", src_h, src_w, h, w);
  const FlatGeom g = flat_geom(n, h, w);
  if (dst_slab4 == nullptr && c % 8 == 0) {
    const long total8 = (long)n * (c / 8) * src_h * src_w;
    int grid8 = ceil_div(total8, 256);
    if (grid8 > 148 * 8) grid8 = 148 * 8;
    flat_from_nchw_vec8_kernel<<<grid8, 256, 0, stream>>>(src, c, src_h, src_w, mode, (__nv_bfloat16*)dst_slab8, scale, g);
    return check_launch("flat_from_nchw_vec8_kernel");
  }
  const long total = (long)n * ((c + 3) / 4) * src_h * src_w;
  int grid = ceil_div(total, 256);
  if (grid > 148 * 8) grid = 148 * 8;
  flat_from_nchw_kernel<<<grid, 256, 0, stream>>>(src, c, src_h, src_w, mode, (__nv_bfloat16*)dst_slab8, dst_slab4, scale, g);
  return check_launch("flat_from_nchw_kernel");
}

extern "C" int dbm_flat_to_nchw_ex(const float* src_slab4, const void* src_slab8, float* dst, int c, int dst_h, int dst_w,
                                   int mode, int n, int h, int w, cudaStream_t stream) {
  DBM_REQUIRE((src_slab4 != nullptr) != (src_slab8 != nullptr) && dst, "flat_to_nchw: exactly one source expected");
  if (mode == 0) DBM_REQUIRE(dst_h <= h && dst_w <= w, "flat_to_nchw: %dx%d window exceeds %dx%d", dst_h, dst_w, h, w);
  else DBM_REQUIRE((dst_h + 1) / 2 <= h && (dst_w + 1) / 2 <= w, "flat_to_nchw: depth-to-space %dx%d exceeds %dx%d", dst_h, dst_w, h, w);
  const FlatGeom g = flat_geom(n, h, w);
  const int cg = src_slab4 ? 4 : 8;
  if (c % cg == 0) {
    const long totalv = (long)n * (c / cg) * dst_h * dst_w;
    int gridv = ceil_div(totalv, 256);
    if (gridv > 148 * 8) gridv = 148 * 8;
    if (src_slab4) flat_to_nchw_vec_kernel<4><<<gridv, 256, 0, stream>>>(src_slab4, dst, c, dst_h, dst_w, mode, g);
    else flat_to_nchw_vec_kernel<8><<<gridv, 256, 0, stream>>>(src_slab8, dst, c, dst_h, dst_w, mode, g);
    return check_launch("flat_to_nchw_vec_kernel");
  }
  const long total = (long)n * c * dst_h * dst_w;
  int grid = ceil_div(total, 256);
  if (grid > 148 * 8) grid = 148 * 8;
  flat_to_nchw_kernel<<<grid, 256, 0, stream>>>(src_slab4, (const __nv_bfloat16*)src_slab8, dst, c, dst_h, dst_w, mode, g);
  return check_launch("flat_to_nchw_kernel");
}

extern "C" int dbm_flat_from_nchw(const float* src, int c, void* dst_slab8, float* dst_slab4, float scale, int n, int h,
                                  int w, cudaStream_t stream) {
  return dbm_flat_from_nchw_ex(src, c, h, w, 0, dst_slab8, dst_slab4, scale, n, h, w, stream);
}

extern "C" int dbm_flat_to_nchw(const float* src_slab4, const void* src_slab8, float* dst, int c, int n, int h, int w,
                                cudaStream_t stream) {
  return dbm_flat_to_nchw_ex(src_slab4, src_slab8, dst, c, h, w, 0, n, h, w, stream);
}
