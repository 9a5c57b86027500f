/*
 * deepbedmap_b200 -- C ABI of the B200-native ESRGAN hot path of weiji14/deepbedmap.
 *
 * The reference has no FFI: its hot path is a Python/Chainer class surface
 * (GeneratorModel / DiscriminatorModel / loss + step functions in srgan_train.py, the tiler in
 * deepbedmap.py) whose arithmetic is executed by Chainer function nodes. Each entry point
 * below is the drop-in for one group of those nodes; the Python shim in deepbedmap_b200/
 * (model.py, train.py, tiler.py) composes them with the reference's own call surface.
 * See INTEGRATION.md for the binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 (DBM_OK) or a negative status; dbm_last_error() gives the text;
 *     no exceptions cross the ABI;
 *   - all pointers are DEVICE pointers owned by the caller unless named host_*; no allocation
 *     happens inside the library; all work is enqueued on the caller's `stream`;
 *   - tensors at the boundary are float32, NCHW, C-contiguous (Chainer layout). A
 *     `*_batch_stride` argument (elements; 0 = dense) lets a call read or write a channel slice
 *     of a wider NCHW buffer, which is how F.concat (srgan_train.py:341-353) is realised
 *     without copies;
 *   - "slab8" = bf16 [N][C/8][H][W][8], "slab4" = fp32 [N][C/4][H][W][4]: the tensor-core
 *     path's internal HBM layouts (one 16-byte vector per pixel per slab).
 */
#ifndef DEEPBEDMAP_B200_H_
#define DEEPBEDMAP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define DBM_OK 0
#define DBM_ERR_INVALID (-1)
#define DBM_ERR_CUDA (-2)

int dbm_version(void);
long dbm_launch_count(void); /* kernels this library has launched since it was loaded (bench.py reports the difference) */
const char* dbm_last_error(void);
/* Deterministic training arithmetic (the reference sets chainer.global_config.cudnn_deterministic = True,
 * srgan_train.py:69): with on != 0 every reduction that otherwise combines partial sums with floating-point atomics
 * runs in a fixed order -- single-contributor launches for split-K / batch-reduced weight and bias gradients, exact
 * 64-bit fixed-point accumulation for the deformable layers' scatter (the library then owns a grow-only device scratch
 * of 8 bytes per scattered element). Two runs of the same steps give bit-identical weights; slower. Default off. */
int dbm_set_deterministic(int on);
/* Persistent kernels of the TRAINING step (weight gradients) leave `n` SMs to concurrently running streams (the
 * discriminator chain on its high-priority stream); results do not depend on it. Default 0. */
int dbm_set_sm_reserve(int n);

/* ---- fp32 convolution family -------------------------------------------------------------
 * L.Convolution2D forward (+ optional fused F.leaky_relu(slope=0.2)):
 *   srgan_train.py:223-254 (stem: k3s1p0, k30s10p0, k6s2p0), :292-331, :467-503 (k3s1p1),
 *   :617-634 (discriminator: k3s1p1, k4s2p1). Supported (ksize, stride): (3,1) (4,2) (6,2) (30,10).
 * The two gradient entry points replace Chainer's autograd of the same link
 * (d_loss.backward() / g_loss.backward(), srgan_train.py:1163, 1256). */
int dbm_conv2d_fwd_f32(const float* x, long x_batch_stride, const float* w, const float* bias, float* y,
                       long y_batch_stride, int n, int c, int h, int wd, int o, int ksize, int stride, int pad,
                       int act, cudaStream_t stream);
int dbm_conv2d_bwd_data_f32(const float* dy, long y_batch_stride, const float* w, float* dx, long x_batch_stride,
                            int n, int c, int h, int wd, int o, int ksize, int stride, int pad, int accumulate,
                            cudaStream_t stream);
/* dw += ...  (caller zeroes the gradient buffer once per step: Link.cleargrads(), :1162, 1255) */
int dbm_conv2d_bwd_weight_f32(const float* x, long x_batch_stride, const float* dy, long y_batch_stride, float* dw,
                              int n, int c, int h, int wd, int o, int ksize, int stride, int pad,
                              cudaStream_t stream);
int dbm_bias_grad_f32(const float* dy, long dy_batch_stride, float* db, int n, int o, int hw, cudaStream_t stream);

/* Batched strided GEMM: L.Linear (srgan_train.py:646-647, 694-696), the filter contraction of the
 * deformable convolution, and their gradients. accumulate: 0 overwrite, 1 +=, 2 atomicAdd. */
int dbm_gemm_f32(const float* a, long lda_m, long lda_k, long a_batch_stride, const float* b, long ldb_k, long ldb_n,
                 long b_batch_stride, float* c, long ldc_m, long ldc_n, long c_batch_stride, const float* bias, int m,
                 int n, int k, int batch, int act, int accumulate, cudaStream_t stream);
/* Same contract, operands rounded to bf16 on the fly, fp32 accumulation on the tensor cores (the contractions of the
 * deformable layer on the bf16 training path, srgan_train.py:506-514). accumulate: 0 overwrite, 2 atomic batch sum. */
int dbm_gemm_bf16(const float* a, long lda_m, long lda_k, long a_batch_stride, const float* b, long ldb_k, long ldb_n,
                  long b_batch_stride, float* c, long ldc_m, long ldc_n, long c_batch_stride, const float* bias, int m,
                  int n, int k, int batch, int act, int accumulate, cudaStream_t stream);

/* ---- element-wise / layout ------------------------------------------------------------------ */
/* out = a*x + b*y on (batch, inner) views: F.add(a5 * residual_scaling, a0), srgan_train.py:358, 402, 551 */
int dbm_axpby_f32(const float* x, long x_bs, const float* y, long y_bs, float* out, long out_bs, float a, float b,
                  int nbatch, long inner, cudaStream_t stream);
int dbm_lrelu_fwd_f32(const float* x, float* y, long total, cudaStream_t stream);
/* backward of F.leaky_relu given its output y: dx (+)= dy * (y >= 0 ? 1 : 0.2) */
int dbm_lrelu_bwd_f32(const float* dy, long dy_bs, const float* y, long y_bs, float* dx, long dx_bs, int nbatch,
                      long inner, int accumulate, cudaStream_t stream);
/* F.resize_images(mode="nearest") to 2x (srgan_train.py:556-566) and its adjoint */
int dbm_upsample2_fwd_f32(const float* x, float* y, long planes, int h, int w, cudaStream_t stream);
int dbm_upsample2_bwd_f32(const float* dy, float* dx, long planes, int h, int w, cudaStream_t stream);
int dbm_fill_f32(float* p, float v, long n, cudaStream_t stream);
int dbm_nchw_to_slab8(const float* src, long src_batch_stride, void* dst_slab8, int n, int c, int h, int w,
                      int dst_cs_total, int dst_cs0, cudaStream_t stream);
int dbm_slab8_to_nchw(const void* src_slab8, int src_cs_total, int src_cs0, float* dst, long dst_batch_stride, int n,
                      int c, int h, int w, cudaStream_t stream);
int dbm_nchw_to_slab4(const float* src, long src_batch_stride, float* dst_slab4, int n, int c, int h, int w,
                      cudaStream_t stream);
int dbm_slab4_to_nchw(const float* src_slab4, float* dst, long dst_batch_stride, int n, int c_slab, int c_keep, int h,
                      int w, cudaStream_t stream);
/* split-bf16 operand buffers of dbm_trunk_umma_split: v = hi + lo (two bf16 terms), slabs per 16 channels
 * [hi a | hi b | lo a | lo b] (2 * c / 8 slabs per image); and the trunk kernels' fp32 slab8f [N][C/8][H][W][8] -> NCHW */
int dbm_nchw_to_slab8_split(const float* src, long src_batch_stride, void* dst_slab8_split, int n, int c, int h, int w,
                            cudaStream_t stream);
int dbm_slab8f_to_nchw(const float* src_slab8f, float* dst, long dst_batch_stride, int n, int c, int h, int w,
                       cudaStream_t stream);

/* ---- tensor-core trunk: 3x3 'same' conv, tcgen05 implicit GEMM ---------------------------------
 * Replaces L.Convolution2D(k3,s1,p1) + F.leaky_relu + F.concat + (x*beta, F.add) +
 * F.resize_images(nearest) chains of srgan_train.py:339-358, 397-402, 541-568 and the
 * offset_conv of L.DeformableConvolution2D (:506-523).
 *   v = conv(in[:, :cin]) + bias;  if res1: v = res1 + beta*v;  if res2: v = res2 + beta*v;
 *   if act: v = lrelu(v);  out_f32_slab4[.., cs0..] = v;  out_slab8[.., cs0..] = bf16(v)
 *   (up2: every output pixel is written to its 2x2 nearest-neighbour block of a 2H x 2W map).
 * cout_padded in {32, 64}; cin multiple of 32. Weights come from dbm_pack_conv3x3_weights. */
int dbm_pack_conv3x3_weights(const float* w_oihw, void* packed_bf16, int cout, int cin, int cout_padded, int ck,
                             cudaStream_t stream);
/* Rows [cout0, cout0+cout) of the packed image <- w[o][w_c0 + c][tap] of an (cout, w_cin_total, 3, 3) filter
 * (c < cin); other rows untouched. Stacks several filters that share an input along Cout. */
int dbm_pack_conv3x3_weights_slice(const float* w_oihw, int w_cin_total, int w_c0, void* packed_bf16, int cout,
                                   int cout0, int cin, int cout_padded, int ck, cudaStream_t stream);
/* The same for a whole model in ONE launch: table_dev = num_entries 48-byte records
 * {const float* w; bf16* out; int cout, cout0, cin, w_cin_total, w_c0, cout_padded, ck, mode}
 * (struct PackEntry, csrc/umma_conv3x3.cu); max_elements = the largest 9*cin*cout_padded. */
int dbm_pack_conv3x3_table(const void* table_dev, int num_entries, long max_elements, cudaStream_t stream);
int dbm_conv3x3_umma(const void* in_slab8, int in_cs_total, int cin, const void* wpacked, const float* bias,
                     int cout_padded, int n, int h, int w, float beta, int act, int up2, void* out_slab8,
                     int out_cs_total, int out_cs0, float* out_f32_slab4, int out_f32_cs_total, int out_f32_cs0,
                     const float* res1_slab4, const float* res2_slab4, cudaStream_t stream);

/* Persistent whole-trunk kernel: pre-residual conv + 3*nb residual dense blocks + post-residual conv
 * (srgan_train.py:541-551) in ONE launch; `layers_dev` is a device array of `num_layers` 128-byte records
 * (struct TrunkLayer in csrc/umma_trunk.cu: weight/bias/output/residual/stash pointers, cin, cout, input
 * buffer id {0 = stem_slab8, 1 = cat_a, 2 = cat_b} and first input slab, epilogue flags). A record is one
 * MMA pass; with dense-block pairing (model.py) a pass computes one layer plus the partial sums of the
 * next layer over their shared inputs. flags_dev holds
 * num_layers * n * ceil(h/32) * ceil(w/16) uint32 (zeroed by the call). */
int dbm_trunk_umma(const void* layers_dev, int num_layers, int n, int h, int w, const void* stem_slab8,
                   int stem_cs_total, const void* cat_a_slab8, const void* cat_b_slab8, int cat_cs_total,
                   unsigned int* flags_dev, cudaStream_t stream);
/* The same pass table in split-bf16 arithmetic (GeneratorModel(precision="bf16x3")): the reference computes these
 * convolutions in fp32 (srgan_train.py:339-358); here every activation and filter is carried as two bf16 terms and each
 * 16-channel K chunk is contracted three times (x_hi w_hi + x_lo w_hi + x_hi w_lo, fp32 accumulation): fp32-grade
 * results on the bf16 tensor pipe at three times the MMA work. Buffers hold 2 x cs_total slabs (layout above), filters
 * are packed by dbm_pack_conv3x3_table entries with mode bit 16; the cs / channel fields of the table stay logical. */
int dbm_trunk_umma_split(const void* layers_dev, int num_layers, int n, int h, int w, const void* stem_slab8,
                         int stem_cs_total, const void* cat_a_slab8, const void* cat_b_slab8, int cat_cs_total,
                         unsigned int* flags_dev, cudaStream_t stream);

/* ---- tensor-core TRAINING trunk ("flat-padded" layout, csrc/umma_flat.cu) --------------------------
 * Forward, data gradient and weight gradient of the trunk's L.Convolution2D(k3,s1,p1) links
 * (srgan_train.py:292-358, 467-486) and of their autograd in g_loss.backward() (:1256) as tcgen05
 * implicit GEMMs. Activations / gradients live in flat slabs: every image keeps its one-pixel zero
 * border and the padded images are flattened, p = (img*(h+2) + y)*(w+2) + x;
 *   bf16 slab8 [C/8][Pg][8], fp32 slab4 [C/4][Pg][4]; dbm_flat_geometry -> {P, tiles, G0, Pg, R}:
 *   Pg = slab stride in positions, G0 = leading zero guard. Buffers must be zero-initialised once;
 *   the kernels only ever write interior positions.
 * dbm_flat_conv3x3_seq runs `count` launches described by 472-byte HOST records (struct FlatLaunch:
 *   {const bf16* in; const bf16* wpacked; int cin, nout, ny, pad; long w_chunk_stride; FlatEpiBlock blk[6]}),
 *   each a 3x3 'same' conv with ny chunks (grid.y) of N = nout in {32..192} output columns (chunk y reads
 *   filter image y and advances every epilogue pointer by y*N channels); only rows/columns 1..out_h/out_w of
 *   the interior are written (0 = all). The epilogue is given per 32 columns by a 72-byte
 *   FlatEpiBlock {bias, add1, add2, mask, out_f32, out_bf16 (pointers to the block's first slab),
 *   s1, beta, beta2, out_scale, act}:
 *     v = acc + bias; v = s1*add1 + beta*v; v = add2 + beta2*v; act: v = lrelu(v);
 *     mask: v *= (mask >= 0 ? 1 : 0.2); out_f32 = v; out_bf16 = bf16(out_scale*v).
 *   Forward filters are packed by dbm_pack_conv3x3_table with ck = 16; data-gradient filters with
 *   PackEntry.mode = 1 (transposed + flipped).
 * dbm_flat_wgrad: dW[o][c][tap] partial sums; units_dev = 48-byte records {const bf16* act; const bf16*
 *   gout; float* partial[9][32][128]; int blk0, nblk, nslab; pad} (struct WgradUnit);
 * dbm_flat_wgrad_reduce: 48-byte records {const float* partial; float* dw; long split_stride; int nsplit,
 *   cin_total, c0, o0, nch, mode}: dw[(o0+o)*cin_total + c0 + c][tap] += sum_s partial[s][tap][o][c];
 * dbm_flat_bias_grad: 16-byte records {const bf16* gout; float* db}: db[0:32] += sum_p gout[.][p]. */
int dbm_flat_geometry(int n, int h, int w, int* out5_host);
int dbm_flat_conv3x3_seq(const void* launches_host, int count, int n, int h, int w, int out_h, int out_w,
                         cudaStream_t stream);
/* The same launch list as ONE persistent launch: layer l's tile t waits for tiles t-1..t+1 of layer l-1
 * (device flags, count * tiles uint32, zeroed here). launches_dev = device copy of launches_host. */
int dbm_flat_conv3x3_chain(const void* launches_host, const void* launches_dev, int count, int n, int h, int w,
                           int out_h, int out_w, void* flags_dev, cudaStream_t stream);
/* Image-resident trunk forward for small tiles ((h+2)*(w+2) <= 128 flat positions per image): the whole chain
 * pre-residual conv -> residual dense blocks -> post-residual conv in one launch with the activations of an image
 * pair held in shared memory / TMEM (csrc/umma_local.cu). passes_dev: device array of 96-byte LocalPass records
 * (deepbedmap_b200/flat.py LOCAL_PASS_DTYPE); s0_flat: stem output, flat bf16 [16][Pg][8]; x0 / xrr scratch:
 * n * 16 * 128 * 4 floats each. Replaces the same reference ops as dbm_flat_conv3x3_chain's forward table
 * (srgan_train.py:339-358, 397-402, 541-551). */
int dbm_trunk_local_fwd(const void* passes_dev, int count, int n, int h, int w, const void* s0_flat,
                        float* x0_scratch, float* xrr_scratch, cudaStream_t stream);
/* The data-gradient chain of the same trunk (autograd of the links above in g_loss.backward(), srgan_train.py:1256),
 * image-resident: gradients wrt the dense-block slots accumulate in TMEM, the bf16 gradients wrt every conv output
 * are written to the flat buffers dbm_flat_wgrad reads. gpost_flat: bf16(d loss / d a3), flat [8][Pg][8]. */
int dbm_trunk_local_bwd(const void* passes_dev, int count, int n, int h, int w, const void* gpost_flat,
                        float* dxrr_scratch, cudaStream_t stream);
int dbm_flat_wgrad(const void* units_dev, int num_units, int n, int h, int w, cudaStream_t stream);
/* the same with an upper bound on the persistent grid of this launch (0 = none): lets two models' weight-gradient
 * kernels share the SMs side by side */
int dbm_flat_wgrad_ctas(const void* units_dev, int num_units, int n, int h, int w, int max_ctas, cudaStream_t stream);
int dbm_flat_wgrad_reduce(const void* entries_dev, int count, cudaStream_t stream);
int dbm_flat_bias_grad(const void* entries_dev, int count, int n, int h, int w, cudaStream_t stream);
/* NCHW fp32 (n, c, h, w) -> scale * x into a flat slab8 and/or slab4 (either may be NULL), and back.
 * _ex: mode 0 = the (src_h, src_w) image sits in the top-left corner of the (h, w) interior; mode 1 = space-to-depth
 * by 2 (pixel (y, x) of channel c -> channel ((y&1)*2 + (x&1))*C + c at (y>>1, x>>1)): with PackEntry.mode 2 / 3
 * filters the 4x4 stride-2 pad-1 convolutions of the discriminator (srgan_train.py:626-634) run as 3x3 GEMMs. */
int dbm_flat_from_nchw_ex(const float* src, int c, int src_h, int src_w, int mode, void* dst_slab8, float* dst_slab4,
                          float scale, int n, int h, int w, cudaStream_t stream);
int dbm_flat_to_nchw_ex(const float* src_slab4, const void* src_slab8, float* dst, int c, int dst_h, int dst_w, int mode,
                        int n, int h, int w, cudaStream_t stream);
int dbm_flat_from_nchw(const float* src, int c, void* dst_slab8, float* dst_slab4, float scale, int n, int h, int w,
                       cudaStream_t stream);
int dbm_flat_to_nchw(const float* src_slab4, const void* src_slab8, float* dst, int c, int n, int h, int w,
                     cudaStream_t stream);

/* ---- fused generator input block for the tensor-core path (DeepbedmapInputBlock.forward,
 * srgan_train.py:256-266): four valid strided convs + F.concat, fp32 math, 128-channel bf16 slab8 out.
 * Filters are passed tap-major (dbm_transpose_f32 of the (32, taps) Chainer filters):
 * w1_filter_tapmajor [900][32]; small_filters_tapmajor [9 | 72 | 9][32] = conv_on_X | conv_on_W2 | conv_on_W3;
 * bias128 = biases of X | W1 | W2 | W3. */
int dbm_transpose_f32(const float* src, float* dst, int rows, int cols, cudaStream_t stream);
int dbm_stem_fwd_slab8(const float* x, const float* w1, const float* w2, const float* w3,
                       const float* w1_filter_tapmajor, const float* small_filters_tapmajor, const float* bias128,
                       void* out_slab8, int out_cs_total, int out_cs0, int n, int h, int w, cudaStream_t stream);
/* conv_on_W1 (1 -> 32, k30 s10 p0, srgan_train.py:231, 259) on the tensor cores: a k30 s10 convolution is a 3x3
 * valid convolution over the 10x10 space-to-depth of its input. With w1 == NULL (and w1_filter_tapmajor == NULL)
 * dbm_stem_fwd_slab8 computes conv_on_X / W2 / W3 only (slabs 0-3, 8-15 of the output); slabs 4-7 then come from
 *   dbm_stem_w1_s2d        w1 (n,1,10h,10w) fp32 -> split operand, bf16 slab8 (n, 40 slabs, h, w):
 *                          channels [x_hi(100->104) | x_lo(104) | x_hi(104) | 0(8)], x = x_hi + x_lo to 2^-18;
 *   dbm_pack_stem_w1       filter (32,1,30,30) fp32 -> UMMA operand image (9*320*32 bf16) [w_hi | w_hi | w_lo | 0];
 *   dbm_conv3x3_umma_valid 3x3 valid conv, 32 output channels, + bias -> bf16 slab8 slot (n, h-2, w-2).
 * fp32-grade accuracy for metre-valued REMA inputs (only the x_lo*w_lo term is dropped). */
int dbm_stem_w1_s2d(const float* w1, void* s2d_slab8, int n, int h, int w, cudaStream_t stream);
int dbm_pack_stem_w1(const float* w1_filter, void* packed_bf16, cudaStream_t stream);
int dbm_conv3x3_umma_valid(const void* in_slab8, int in_cs_total, int cin, const void* wpacked, const float* bias,
                           int n, int h_in, int w_in, void* out_slab8, int out_cs_total, int out_cs0,
                           cudaStream_t stream);
/* Same fused input block, written in the flat-padded layout [16][Pg][8] (geometry of dbm_flat_geometry(n, h-2, w-2));
 * borders / guards of out_flat must be zero (they are never written). Feeds dbm_trunk_local_fwd on small tiles. */
int dbm_stem_fwd_flat(const float* x, const float* w1, const float* w2, const float* w3, const float* w1_filter_tapmajor,
                      const float* small_filters_tapmajor, const float* bias128, void* out_flat, int n, int h, int w,
                      cudaStream_t stream);

/* ---- deformable convolution, tensor-core inference path (L.DeformableConvolution2D 64->64 and 64->1,
 * srgan_train.py:506-523, 572-574): bilinear gather straight into the UMMA operand layout in SMEM,
 * tcgen05 contraction with the SMEM-resident filter (weights packed with ck = 64), bias + LeakyReLU
 * epilogue; the 64->1 output layer is a CUDA-core dot product with fp32 NCHW output.
 * offset_slab4: fp32 slab4 with >= 18 channels ([0:9] = dx, [9:18] = dy). */
int dbm_deform_conv_umma(const void* x_slab8, const float* offset_slab4, int offset_cs_total,
                         const void* wpacked_ck64, const float* bias, int n, int h, int w, int act, void* out_slab8,
                         int out_cs_total, int out_cs0, const float* next_out1_filter, float* next_out1_proj,
                         cudaStream_t stream);
/* Training-path form (forward of final_conv_layer1 under forward_train): offsets as the fp32 NCHW (n,18,h,w) tensor of
 * the offset convolution, output fp32 NCHW (n,64,h,w) without bf16 storage rounding; same operand rounding as the
 * sampler + bf16 GEMM pair it replaces, no `cols` buffer. */
int dbm_deform_conv_umma_nchw(const void* x_slab8, const float* offset_nchw18, const void* wpacked_ck64,
                              const float* bias, int n, int h, int w, int act, float* out_nchw, cudaStream_t stream);
/* next_out1_filter / next_out1_proj (both or neither): the (1, 64, 3, 3) filter of a FOLLOWING single-output
 * deformable layer and a [n][9][h*w] buffer -- the layer's "tap projection" (see dbm_deform_conv_out1) is then
 * computed in this kernel's epilogue from the outputs in registers; finish that layer with dbm_deform_out1_sample. */
/* cols (n, 64*9, h*w) fp32 for the backward of dbm_deform_conv_umma_nchw: the same bilinear samples, gathered from
 * the same bf16 slab8 input (L.DeformableConvolution2D's weight gradient operand, srgan_train.py:506-523). */
int dbm_deform_sample_slab8_f32(const void* x_slab8, const float* offset_nchw18, float* cols, int n, int h, int w,
                                cudaStream_t stream);
int dbm_deform_out1_sample(const float* proj, const float* offset_slab4, int offset_cs_total, const float* bias,
                           float* y, int n, int h, int w, cudaStream_t stream);
/* proj_scratch: n*9*h*w floats (the 64 channels projected onto the 9 taps before sampling) */
int dbm_deform_conv_out1(const void* x_slab8, const float* offset_slab4, int offset_cs_total, const float* w_f32,
                         const float* bias, float* y, float* proj_scratch, int n, int h, int w, cudaStream_t stream);

/* ---- deformable convolution, fp32 path (L.DeformableConvolution2D, srgan_train.py:506-523) -----
 * cols[n][c*9+t][pixel] = bilinear sample; contraction with W (O, C*9) is a dbm_gemm_f32 call.
 * offset: (N,18,H,W), channels [0:9] = dx, [9:18] = dy of tap t = ky*3+kx. */
int dbm_deform_sample_f32(const float* x, const float* offset, float* cols, int n, int c, int h, int w,
                          cudaStream_t stream);
/* dx += scatter(dcols) (may be NULL), doffset = d/d(offset) */
int dbm_deform_bwd_f32(const float* x, const float* offset, const float* dcols, float* dx, float* doffset, int n,
                       int c, int h, int w, cudaStream_t stream);

/* Single-output deformable layer (final_conv_layer2, 64 -> 1; srgan_train.py:515-523, 574) by tap projection:
 * proj[n][t] = sum_c W[0,c,t] x[n][c] (kept for backward), y = bias + sum_t bilinear(proj[t], tap position).
 * Backward: dw (1,C,3,3) accumulated, dx written (or accumulated), doffset (N,18,H,W) written;
 * dproj_scratch = N*9*H*W floats. */
int dbm_deform1_fwd_f32(const float* x, const float* offset, const float* w, const float* bias, float* y, float* proj,
                        int n, int c, int h, int w_, cudaStream_t stream);
int dbm_deform1_bwd_f32(const float* x, const float* offset, const float* w, const float* proj, const float* dy,
                        float* dw, float* dx, int accumulate_dx, float* doffset, float* dproj_scratch, int n, int c,
                        int h, int w_, cudaStream_t stream);

/* ---- discriminator normalisation (L.BatchNormalization + F.leaky_relu, srgan_train.py:636-689) - */
int dbm_bn_lrelu_fwd_f32(const float* x, float* y, const float* gamma, const float* beta, float* avg_mean,
                         float* avg_var, float* save_mean, float* save_invstd, int n, int c, int hw, float eps,
                         float decay, int train, cudaStream_t stream);
int dbm_bn_lrelu_bwd_f32(const float* x, const float* y, const float* dy, float* dx, const float* gamma,
                         const float* save_mean, const float* save_invstd, float* dgamma, float* dbeta,
                         float* scratch2c, int n, int c, int hw, cudaStream_t stream);
/* `groups` independent BatchNormalization (+ LeakyReLU) passes over a batch stacked along N in one pair of launches
 * (the discriminator step's D(real) | D(fake), srgan_train.py:1145-1146): x, y (groups * n, c, hw); save_mean /
 * save_invstd [groups][c]; running statistics updated group after group; backward scratch [groups][2 c]. Values equal
 * `groups` consecutive single-group calls bit for bit. */
int dbm_bn_lrelu_fwd_groups_f32(const float* x, float* y, const float* gamma, const float* beta, float* avg_mean,
                                float* avg_var, float* save_mean, float* save_invstd, int groups, int n, int c, int hw,
                                float eps, float decay, int train, cudaStream_t stream);
int dbm_bn_lrelu_bwd_groups_f32(const float* x, const float* y, const float* dy, float* dx, const float* gamma,
                                const float* save_mean, const float* save_invstd, float* dgamma, float* dbeta,
                                float* scratch, int groups, int n, int c, int hw, cudaStream_t stream);

/* ---- losses (srgan_train.py:841-1009) -------------------------------------------------------- */
/* out2[0] = RaGAN loss (calculate_discriminator_loss), out2[1] = F.binary_accuracy of
 * [real; fake] against [1; 0]; d_real/d_fake (nullable) = grad_scale * dLoss/dlogit. */
int dbm_ragan_loss_f32(const float* real_pred, const float* fake_pred, int n, float t_real_minus_fake,
                       float t_fake_minus_real, float grad_scale, float* out2, float* d_real, float* d_fake,
                       cudaStream_t stream);
/* sums4 = {sum|yp-yt|, sum|avgpool4(yp)-x_topo|, sum ssim_map, sum (yp-yt)^2};
 * dy (nullable) = d/dyp of w_content*L1 + w_topo*Topo + w_struct*(1 - SSIM). */
int dbm_gen_image_loss_f32(const float* y_pred, const float* y_true, const float* x_topo, int n, int h, int w,
                           float w_content, float w_topo, float w_struct, float* sums4, float* dy,
                           cudaStream_t stream);

/* ---- chainer.optimizers.Adam(alpha, beta1, beta2, eps) over a flat parameter buffer (:1043-1048) */
int dbm_adam_step_f32(float* params, const float* grads, float* m, float* v, long n, float alpha, float beta1,
                      float beta2, float eps, int t, float grad_scale, cudaStream_t stream);
/* Same update with the step count t kept on the device (incremented here, before the update): the form a CUDA-graph
 * replay of the training step needs -- a host-side t would freeze the bias correction into the graph. */
int dbm_adam_step_dev_f32(float* params, const float* grads, float* m, float* v, long n, float alpha, float beta1,
                          float beta2, float eps, int* t_dev, float grad_scale, cudaStream_t stream);

/* ---- continent tiler staging (deepbedmap.py:663-665, 715-722, 731-736) ------------------------- */
int dbm_crop_clip_f32(const float* src, int hs, int ws, float* dst, int c, int y0, int x0, int h, int w, int clip0,
                      cudaStream_t stream);
int dbm_place_tile_f32(const float* tile, int th, int tw, int cy, int cx, float* canvas, int ch, int cw, int ys,
                       int xs, int hh, int ww, cudaStream_t stream);

/* Y_hat.astype(np.int16) on the device (deepbedmap.py:751): C-cast semantics of NumPy on x86-64
 * (truncate toward zero to int32, NaN / out-of-range -> INT_MIN, keep the low 16 bits: NaN -> 0). */
int dbm_f32_to_i16(const float* src, void* dst_i16, long n, cudaStream_t stream);

/* Strided 2-D copy (cudaMemcpy2DAsync, kind inferred from the pointers): `rows` rows of `width_bytes`, pitches in
 * bytes. The tiler streams every finished tile row of its device canvas into the caller's pinned (or
 * cudaHostRegister-ed shared) host DEM with it while later tiles compute (Y_hat[:, y_slice, x_slice] = ...,
 * deepbedmap.py:733-736). dst / src may be host or device pointers. */
int dbm_copy2d_async(void* dst, size_t dst_pitch, const void* src, size_t src_pitch, size_t width_bytes, size_t rows,
                     cudaStream_t stream);

/* ---- on-device minibatch assembly (chainer SerialIterator + concat_examples, srgan_train.py:132-166):
 * dst[j, :] = src[index[j], :] for j < nrows; rows of `row` floats; index = int64 on the device. */
int dbm_gather_rows_f32(const float* src, long src_rows, const long* index_dev, float* dst, long row, int nrows,
                        cudaStream_t stream);

/* ---- model-level entry points: GeneratorModel (srgan_train.py:421-576) without the Python shim ------------
 * A host in any language runs the generator's inference forward with
 *     dbm_gen_create -> dbm_gen_set_param (every array of the Chainer .npz, keys of SURVEY App. C:
 *     dbm_gen_array_info lists them in file order) -> dbm_gen_workspace_bytes -> dbm_gen_forward.
 * The handle owns the fp32 master weights (device; or views a caller-owned flat device buffer of
 * dbm_gen_count_params floats in App. C order, dbm_gen_bind_params), their re-packed bf16 UMMA operand images and
 * the pass table of the persistent trunk kernel -- with the discriminator handle's (below), the only device memory this
 * library allocates besides the deterministic mode's scratch. Activations
 * live in the caller's `workspace` (device, 1024-byte aligned, dbm_gen_workspace_bytes(n, h, w) bytes); everything is
 * enqueued on `stream`. Arithmetic: the tensor-core inference path (bf16 operands, fp32 accumulation, fp32 residual
 * stream; conv_on_W1 as a split-bf16 GEMM) or, after dbm_gen_set_precision(gen, 1), the split-bf16 path;
 * inter_channels 32 or 64, out_channels == 1 as in the reference.
 *   x (n,1,h,w), w1 (n,1,10h,10w), w2 (n,2,2h,2w), w3 (n,1,h,w) fp32 NCHW device -> y_out (n,1,4(h-2),4(w-2)).
 * A handle is bound to the device current at creation and is not thread-safe (one host thread per GPU, as the
 * reference's one process per GPU, srgan_train.py:58-61). The first forward on a new (workspace, shape) uploads the
 * pass table and synchronises the stream once; later calls only enqueue (CUDA-graph capturable). */
typedef struct dbm_gen dbm_gen;
int dbm_gen_create(int num_residual_blocks, float residual_scaling, int inter_channels, dbm_gen** out);
int dbm_gen_destroy(dbm_gen* gen);
long dbm_gen_count_params(const dbm_gen* gen);              /* 8 907 749 for 12 blocks (srgan_train.py:446-447) */
int dbm_gen_num_arrays(const dbm_gen* gen);                 /* 384 for 12 blocks */
int dbm_gen_array_info(const dbm_gen* gen, int index, const char** key, int* ndim, int* dims4, long* flat_offset);
int dbm_gen_set_param(dbm_gen* gen, const char* key, const float* host_values, int ndim, const int* dims);
int dbm_gen_bind_params(dbm_gen* gen, float* device_flat);
int dbm_gen_mark_updated(dbm_gen* gen);                     /* after writing into a bound parameter buffer */
/* precision of dbm_gen_forward: 0 = bf16 tensor-core path (default), 1 = "bf16x3" -- split-bf16 trunk and upsample convs
 * on the tensor cores (dbm_trunk_umma_split), input block and deformable layers on the fp32 kernels: fp32-grade results
 * (the reference computes in fp32). Changes dbm_gen_workspace_bytes; call before sizing the workspace. */
int dbm_gen_set_precision(dbm_gen* gen, int precision);
size_t dbm_gen_workspace_bytes(const dbm_gen* gen, int n, int h, int w);
int dbm_gen_forward(dbm_gen* gen, const float* x, const float* w1, const float* w2, const float* w3, int n, int h,
                    int w, float* y_out, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---- model-level entry points: DiscriminatorModel (srgan_train.py:591-699) without the Python shim ---------------
 * A host in any language runs the discriminator's training forward, backward and BatchNormalization bookkeeping with
 *     dbm_disc_create -> dbm_disc_set_param (every array of the Chainer .npz: dbm_disc_array_info lists the 33
 *     parameters in flat-buffer order, then avg_mean / avg_var / N of batch_norm1..9) -> dbm_disc_workspace_bytes ->
 *     per step: dbm_disc_zero_grads -> dbm_disc_forward(train = 1, save = 1) -> loss gradient -> dbm_disc_backward.
 * The handle owns the fp32 master weights and gradients (device; or views caller-owned flat device buffers of
 * dbm_disc_count_params floats in layout.discriminator_shapes() order, dbm_disc_bind_params / dbm_disc_bind_grads: how
 * an optimizer such as dbm_adam_step_f32 reaches them), the running statistics (device) and the nine N counters (host,
 * kept as loaded: Chainer counts only in finetune mode, which the reference never enters), the packed bf16 operand
 * images of conv_layer1..9 and every device table. x (n,1,36,36), logits (n,1), dlogit (n,1), the workspace (device,
 * 1024-byte aligned, dbm_disc_workspace_bytes(n) bytes) and the stream belong to the caller.
 *   forward: `groups` independent BatchNormalization batches stacked along n (D(real) | D(fake), srgan_train.py:
 *     1145-1146; n % groups == 0); train = 1: batch statistics, running statistics updated group after group
 *     (eps 1e-5, decay 0.9); train = 0: running statistics. save = 1 (needs train = 1) keeps in the workspace what
 *     backward needs; a later forward on the same workspace discards it.
 *   backward: accumulates d(loss)/d(params) into the gradient buffer (Chainer semantics: zero it per step) for the saved
 *     pass of that workspace, and consumes it. Two passes in flight = two workspaces.
 * Arithmetic: precision 0 (default) = conv_layer1..9 on the tcgen05 tensor cores (bf16 operands, fp32 accumulation;
 * DiscriminatorModel(precision="bf16")), 1 = fp32 CUDA-core convolutions ("fp32"); conv_layer0, BatchNormalization,
 * LeakyReLU and the Linear layers are fp32 in both. Results equal the Python class's bit for bit (gradients: under
 * dbm_set_deterministic(1)). The first forward on a new (workspace, n, precision) uploads its tables and synchronises
 * the stream once; later calls only enqueue (CUDA-graph capturable). A handle is bound to the device current at
 * creation and is not thread-safe. dbm_disc_get_param / _set_param copy synchronously (no stream). */
typedef struct dbm_disc dbm_disc;
int dbm_disc_create(dbm_disc** out);
int dbm_disc_destroy(dbm_disc* disc);
/* 0 = bf16 tensor-core convolutions (default), 1 = fp32; changes dbm_disc_workspace_bytes and drops saved passes */
int dbm_disc_set_precision(dbm_disc* disc, int precision);
long dbm_disc_count_params(const dbm_disc* disc);           /* 10 370 761 (srgan_train.py:607-608) */
int dbm_disc_num_arrays(const dbm_disc* disc);              /* 60: 33 parameters + 27 BatchNormalization persistents */
/* flat_offset: position in the parameter buffer, -1 for the persistents; N has ndim 0 */
int dbm_disc_array_info(const dbm_disc* disc, int index, const char** key, int* ndim, int* dims4, long* flat_offset);
int dbm_disc_set_param(dbm_disc* disc, const char* key, const float* host_values, int ndim, const int* dims);
int dbm_disc_get_param(const dbm_disc* disc, const char* key, float* host_values);   /* parameters and persistents */
int dbm_disc_bind_params(dbm_disc* disc, float* device_flat);
int dbm_disc_bind_grads(dbm_disc* disc, float* device_flat);   /* drops saved passes */
int dbm_disc_mark_updated(dbm_disc* disc);                  /* after writing into a bound parameter buffer */
int dbm_disc_zero_grads(dbm_disc* disc, cudaStream_t stream);  /* Link.cleargrads(), srgan_train.py:1162 */
size_t dbm_disc_workspace_bytes(const dbm_disc* disc, int n);
int dbm_disc_forward(dbm_disc* disc, const float* x, int n, int groups, int train, int save, float* logits,
                     void* workspace, size_t workspace_bytes, cudaStream_t stream);
int dbm_disc_backward(dbm_disc* disc, const float* dlogit, void* workspace, size_t workspace_bytes, cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DEEPBEDMAP_B200_H_ */
