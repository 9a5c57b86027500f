// Host-built records of the flat-padded tensor-core kernels (csrc/umma_flat.cu): launch records of
// dbm_flat_conv3x3_seq / _chain and the unit / reduction tables of dbm_flat_wgrad / _reduce. Shared by the kernels and
// by the model handles that build these tables in C++ (csrc/disc_api.cu); deepbedmap_b200/flat.py mirrors them.
#pragma once
#include "common.cuh"

namespace dbm {

struct FlatEpiBlock {  // 72 bytes; mirrored by deepbedmap_b200/flat.py (EPI_DTYPE). Pointers are pre-offset to the
  const float* bias;            // block's first slab (fp32: 8 slab4, bf16: 4 slab8); slab stride = Pg positions
  const float* add1;            // v = s1 * add1 + beta * v
  const float* add2;            // v = add2 + beta2 * v
  const __nv_bfloat16* mask;    // v *= (mask >= 0 ? 1 : 0.2)   (LeakyReLU derivative from its bf16 output)
  float* out_f32;
  __nv_bfloat16* out_bf16;      // = bf16(out_scale * v)
  float s1, beta, beta2, out_scale;
  int act, pad;
};
static_assert(sizeof(FlatEpiBlock) == 72, "FlatEpiBlock layout is part of the C ABI");

struct FlatLaunch {  // 472 bytes
  const __nv_bfloat16* in;       // first input slab
  const __nv_bfloat16* wpacked;  // [ny][Cin/16][9][2][N/8][8][8]
  int cin, nout;                 // nout = N = output columns of ONE chunk
  int ny, pad;                   // output-channel chunks (grid.y): chunk y uses filter image y and every epilogue
  long w_chunk_stride;           // pointer advanced by y * N channels; w_chunk_stride = elements per filter image
  FlatEpiBlock blk[6];
};
static_assert(sizeof(FlatLaunch) == 472, "FlatLaunch layout is part of the C ABI");

// Weight gradient: dW[o][c][tap] = sum_p g[o][p] * a[c][p + shift(tap)]   (MN-major operands)
struct WgradUnit {  // 48 bytes; mirrored by flat.py (WGRAD_UNIT_DTYPE)
  const __nv_bfloat16* act;   // first slab of the <= 128-channel input chunk
  const __nv_bfloat16* gout;  // first slab of the 32 output-gradient channels
  float* partial;             // [9][32][128] fp32: partial[tap][o][c]
  int blk0, nblk;             // range of 128-position blocks
  int nslab;                  // input slabs in this chunk (<= 16)
  int tapmask;                // bit t set: tap t is computed (0 = all nine). A 4x4 stride-2 filter embedded as a 3x3
  int pad[2];                 // filter over the four space-to-depth phases has 4 non-zero taps per phase: the other
};                            // five accumulators are neither computed nor written (the reduction skips them too)
static_assert(sizeof(WgradUnit) == 48, "WgradUnit layout is part of the C ABI");

struct WgradReduce {  // 48 bytes; dw[(o0 + o) * cin_total + c0 + c][tap] += sum_s partial[s][tap][o][c]
  const float* partial;
  float* dw;
  long split_stride;  // floats between consecutive splits
  int nsplit, cin_total, c0, o0, nch;
  int mode;           // bits 0-7: 0 = 3x3 filter, 1 = 4x4 stride-2 filter embedded as 3x3 over the 4 space-to-depth
};                    // phases (channel c0 + c = phase * cin_total + cc); bits 8-15: valid output rows (0 = 32)
static_assert(sizeof(WgradReduce) == 48, "WgradReduce layout is part of the C ABI");

}  // namespace dbm
