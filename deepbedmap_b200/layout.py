"""Parameter inventory of the generator / discriminator in the reference's Chainer ``.npz`` key
layout (chainer.serializers.save_npz of the links defined at srgan_train.py:201-699; call sites
srgan_train.py:1355-1361, deepbedmap.py:408), and the generator trunk's pass plan (trunk_plan)."""
from __future__ import annotations

import math
from collections import OrderedDict

import numpy as np

# (out_channels, ksize, stride) of DiscriminatorModel.conv_layer0..9 (srgan_train.py:617-634)
DISC_CONVS = [(64, 3, 1), (64, 4, 2), (128, 3, 1), (128, 4, 2), (128, 3, 1),
              (256, 4, 2), (256, 3, 1), (512, 4, 2), (512, 3, 1), (512, 4, 2)]


def generator_shapes(num_residual_blocks: int = 12, inter_channels: int = 32, out_channels: int = 1):
    g = inter_channels
    s = OrderedDict()
    for name, shp in (("X", (32, 1, 3, 3)), ("W1", (32, 1, 30, 30)), ("W2", (32, 2, 6, 6)), ("W3", (32, 1, 3, 3))):
        s[f"input_block/conv_on_{name}/W"] = shp
        s[f"input_block/conv_on_{name}/b"] = (32,)
    s["pre_residual_conv_layer/W"] = (64, 128, 3, 3)
    s["pre_residual_conv_layer/b"] = (64,)
    for i in range(num_residual_blocks):
        for r in (1, 2, 3):
            p = f"residual_network/{i}/residual_dense_block{r}"
            for k in (1, 2, 3, 4):
                s[f"{p}/conv_layer{k}/W"] = (g, 64 + (k - 1) * g, 3, 3)
                s[f"{p}/conv_layer{k}/b"] = (g,)
            s[f"{p}/conv_layer5/W"] = (64, 64 + 4 * g, 3, 3)
            s[f"{p}/conv_layer5/b"] = (64,)
    for name in ("post_residual_conv_layer", "post_upsample_conv_layer_1", "post_upsample_conv_layer_2"):
        s[f"{name}/W"] = (64, 64, 3, 3)
        s[f"{name}/b"] = (64,)
    for name, oc in (("final_conv_layer1", 64), ("final_conv_layer2", out_channels)):
        s[f"{name}/offset_conv/W"] = (18, 64, 3, 3)
        s[f"{name}/offset_conv/b"] = (18,)
        s[f"{name}/deform_conv/W"] = (oc, 64, 3, 3)
        s[f"{name}/deform_conv/b"] = (oc,)
    return s


def discriminator_shapes():
    s = OrderedDict()
    cin = 1
    for i, (cout, k, _) in enumerate(DISC_CONVS):
        s[f"conv_layer{i}/W"] = (cout, cin, k, k)
        if i == 0:
            s["conv_layer0/b"] = (cout,)
        else:
            s[f"batch_norm{i}/gamma"] = (cout,)
            s[f"batch_norm{i}/beta"] = (cout,)
        cin = cout
    s["linear_1/W"] = (100, 512)
    s["linear_1/b"] = (100,)
    s["linear_2/W"] = (1, 100)
    s["linear_2/b"] = (1,)
    return s


def discriminator_persistents():
    """avg_mean / avg_var / N of every L.BatchNormalization (serialised with the params)."""
    s = OrderedDict()
    for i, (cout, _, _) in enumerate(DISC_CONVS):
        if i:
            s[f"batch_norm{i}/avg_mean"] = (cout,)
            s[f"batch_norm{i}/avg_var"] = (cout,)
    return s


def he_normal(rng: np.random.RandomState, shape, scale: float = 0.1) -> np.ndarray:
    """chainer.initializers.HeNormal(scale=0.1, fan_option="fan_in") (srgan_train.py:220)."""
    fan_in = int(np.prod(shape[1:]))
    return rng.normal(0.0, scale * math.sqrt(2.0 / fan_in), size=shape).astype(np.float32)


def init_values(shapes, seed: int, scale: float = 0.1):
    rng = np.random.RandomState(seed)
    out = OrderedDict()
    for k, shp in shapes.items():
        if k.endswith("/W"):
            out[k] = he_normal(rng, shp, scale)
        elif k.endswith("/gamma"):
            out[k] = np.ones(shp, np.float32)
        else:
            out[k] = np.zeros(shp, np.float32)
    return out


def trunk_pass(image, cin, cout, in_map, bias=None, act=0, beta=0.0, out=None, out_cs0=0, out_f32=None, res1=None,
               res2=None, up2=0, in_cs0=0, cout_main=None, mode=0):
    """One pass of the trunk kernels (csrc/umma_trunk.cu TrunkLayer) with symbolic operands: ``image`` names the packed
    filter image (model._pack's key without its @trunk / @split suffix), ``bias`` the bias key (default ``image/b``);
    ``in_map`` 0 reads the stem output, 1 / 2 the dense-block buffers cat0 / cat1; ``out`` names the bf16 output buffer
    ("cat0", "cat1", "u1", ...) and ``out_f32`` / ``res1`` / ``res2`` the fp32 ones ("a1", "f32_0".."f32_2")."""
    return dict(image=image, bias=f"{image}/b" if bias is None else bias, cin=cin, cout=cout, in_map=in_map,
                in_cs0=in_cs0, act=act, up2=up2, out=out, out_cs0=out_cs0,
                cout_main=cout if cout_main is None else cout_main, beta=beta, mode=mode, out_f32=out_f32, res1=res1,
                res2=res2)


def trunk_plan(num_residual_blocks: int, inter_channels: int, residual_scaling: float, paired: bool,
               paired_convs=(1, 3)):
    """Pass sequence of the generator trunk (srgan_train.py:541-558) as trunk_pass records: the pre-residual conv
    (a1 = lrelu(conv(a0)), kept in fp32), 3 * nb residual dense blocks, then the post-residual conv with the skip a1 and
    the nearest x2 fused (into u1). Dense block j reads and extends cat[j % 2] and writes its output into the other
    buffer; the fp32 residual stream rotates through a ring of three buffers so that a conv5 never writes the block
    input (res1) or, on the third block of an RRDB, the RRDB input (res2) it reads.

    ``paired`` (inter_channels 32 only) fuses conv_k with conv_{k+1} for each k in ``paired_convs`` (1 and / or 3):
      head ("{pre}/pair{k}", mode 1): N = 64 over [a0..a_{k-1}] -> a_k (32 columns, fused epilogue); the other 32
          columns -- the partial sums of conv_{k+1} over the same inputs -- stay in tensor memory
      tail ("{pre}/tail{k+1}", mode 2): N = 32 over a_k only, accumulated onto those columns -> a_{k+1}
    Same FLOPs; 252 N=32 MMAs per 128-pixel tile become 108 N=64 + 36 N=32 MMAs (each MMA re-reads its 4 KB A operand
    from shared memory whatever N is), and nothing but the bf16 features a_k ever leaves the SM. A pair not listed is
    two plain passes."""
    g = inter_channels
    ring = ("f32_0", "f32_1", "f32_2")
    plan = [trunk_pass("pre_residual_conv_layer", 128, 64, 0, act=1, out="cat0", out_f32="a1")]
    cur, cur_f32, fi = 0, "a1", 0
    for i in range(num_residual_blocks):
        rrdb_in = cur_f32
        for r in (1, 2, 3):
            pre = f"residual_network/{i}/residual_dense_block{r}"
            cat = f"cat{cur}"
            for k in (1, 3):
                cin = 64 + (k - 1) * g
                if paired and k in paired_convs:
                    plan.append(trunk_pass(f"{pre}/pair{k}", cin, 64, 1 + cur, bias=f"{pre}/conv_layer{k}/b", act=1,
                                           out=cat, out_cs0=cin // 8, cout_main=32, mode=1))
                    plan.append(trunk_pass(f"{pre}/tail{k + 1}", 32, 32, 1 + cur, bias=f"{pre}/conv_layer{k + 1}/b",
                                           in_cs0=cin // 8, act=1, out=cat, out_cs0=cin // 8 + 4, mode=2))
                else:
                    for kk in (k, k + 1):
                        ci = 64 + (kk - 1) * g
                        plan.append(trunk_pass(f"{pre}/conv_layer{kk}", ci, g, 1 + cur, act=1, out=cat, out_cs0=ci // 8))
            while ring[fi] in (cur_f32, rrdb_in):
                fi = (fi + 1) % 3
            plan.append(trunk_pass(f"{pre}/conv_layer5", 64 + 4 * g, 64, 1 + cur, beta=residual_scaling,
                                   out=f"cat{1 - cur}", out_f32=ring[fi], res1=cur_f32,
                                   res2=rrdb_in if r == 3 else None))
            cur, cur_f32 = 1 - cur, ring[fi]
    plan.append(trunk_pass("post_residual_conv_layer", 64, 64, 1 + cur, beta=1.0, out="u1", res1="a1", up2=1))
    return plan


def infer_num_residual_blocks(keys) -> int:
    """The .npz does not store the block count (the reference gets it from Comet,
    deepbedmap.py:397-405); infer it from the highest residual_network/<i> index."""
    idx = [int(k.split("/")[1]) for k in keys if k.startswith("residual_network/")]
    return max(idx) + 1 if idx else 0
