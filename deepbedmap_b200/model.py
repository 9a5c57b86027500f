"""GeneratorModel / DiscriminatorModel with the reference's call surface
(srgan_train.py:421-576, 591-699), executed by the CUDA kernels of libdeepbedmap_b200.so.

Two arithmetic modes, both on the GPU (there is no CPU path):
  precision="bf16"  inference: trunk / upsample / offset convolutions on the tcgen05 tensor cores
                    (bf16 operands, fp32 TMEM accumulators, fp32 residual stream);
  precision="fp32"  exact float32 CUDA-core path, also the path that keeps activations for
                    backward (the training step).
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Dict, Optional

import numpy as np
import torch

from . import layout, ops
from . import npz as npz_io


# mirror of struct TrunkLayer in csrc/umma_trunk.cu (128 bytes)
TRUNK_LAYER_DTYPE = np.dtype([("wpacked", "<u8"), ("bias", "<u8"), ("out_bf16", "<u8"), ("out_f32", "<u8"),
                              ("res1", "<u8"), ("res2", "<u8"), ("stash_out", "<u8"), ("cin", "<i4"), ("cout", "<i4"),
                              ("in_map", "<i4"), ("in_cs0", "<i4"), ("act", "<i4"), ("up2", "<i4"),
                              ("out_cs_total", "<i4"), ("out_cs0", "<i4"), ("cout_main", "<i4"),
                              ("res1_cs_total", "<i4"), ("beta", "<f4"), ("mode", "<i4"), ("pad", "<i4", (6,))])
assert TRUNK_LAYER_DTYPE.itemsize == 128
# mirror of struct PackEntry in csrc/umma_conv3x3.cu (48 bytes)
PACK_ENTRY_DTYPE = np.dtype([("w", "<u8"), ("out", "<u8"), ("O", "<i4"), ("o0", "<i4"), ("Cin", "<i4"),
                             ("CinTotal", "<i4"), ("c0", "<i4"), ("COUTP", "<i4"), ("CK", "<i4"), ("mode", "<i4")])
assert PACK_ENTRY_DTYPE.itemsize == 48


class Variable:
    """Minimal stand-in for chainer.Variable: callers only use ``.array`` / ``.shape``
    (srgan_train.py:1137, 1229, 1450; deepbedmap.py:421, 733)."""

    def __init__(self, array: torch.Tensor):
        self.array = array
        self.data = array

    @property
    def shape(self):
        return tuple(self.array.shape)

    def numpy(self) -> np.ndarray:
        return self.array.detach().cpu().numpy()


class _DeviceArrayModule:
    """``model.xp`` shim: ``model.xp.asarray(a, dtype="float32")`` moves a host crop to the GPU
    (deepbedmap.py:715-722)."""

    @staticmethod
    def asarray(a, dtype="float32"):
        return as_device(a)


def as_device(a) -> torch.Tensor:
    if isinstance(a, Variable):
        a = a.array
    if isinstance(a, torch.Tensor):
        t = a
    else:
        t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
    return t.to(device="cuda", dtype=torch.float32, non_blocking=True).contiguous()


class _Link:
    """Flat fp32 parameter / gradient buffers on the device with named views."""

    def __init__(self, shapes: "OrderedDict[str, tuple]", values: Dict[str, np.ndarray]):
        if not torch.cuda.is_available():
            raise RuntimeError("deepbedmap_b200 needs a CUDA device (B200); there is no CPU fallback")
        from . import _lib
        _lib.load()  # fail loudly if the CUDA library is missing
        self._shapes = shapes
        total = sum(int(np.prod(s)) for s in shapes.values())
        host = np.empty(total, np.float32)
        self._slices = OrderedDict()
        off = 0
        for k, shp in shapes.items():
            n = int(np.prod(shp))
            host[off:off + n] = np.asarray(values[k], np.float32).reshape(-1)
            self._slices[k] = (off, n)
            off += n
        self.flat = torch.from_numpy(host).cuda()
        self.flat_grad = ops.zeros(total)
        self.p = OrderedDict((k, self.flat[o:o + n].view(shapes[k])) for k, (o, n) in self._slices.items())
        self.g = OrderedDict((k, self.flat_grad[o:o + n].view(shapes[k])) for k, (o, n) in self._slices.items())
        self.version = 0
        self.xp = _DeviceArrayModule()

    # -- chainer.Link surface used by the reference --
    def to_gpu(self, device=None):
        return self

    def params(self):
        return iter(self.p.values())

    def namedparams(self):
        return iter(self.p.items())

    def count_params(self) -> int:
        return int(self.flat.numel())

    def cleargrads(self):
        ops.fill(self.flat_grad, 0.0)

    def set_param(self, key: str, value):
        if key not in self.p:
            raise KeyError(key)
        v = np.asarray(value, np.float32)
        if tuple(v.shape) != tuple(self._shapes[key]):
            raise ValueError(f"{key}: shape {v.shape} != {self._shapes[key]}")
        self.p[key].copy_(torch.from_numpy(np.ascontiguousarray(v)))
        self.version += 1

    def get_param(self, key: str) -> np.ndarray:
        return self.p[key].detach().cpu().numpy()

    def state_dict(self) -> "OrderedDict[str, np.ndarray]":
        return OrderedDict((k, self.get_param(k)) for k in self.p)

    def mark_updated(self):
        self.version += 1

    def grad_range(self, prefixes):
        """[lo, hi) element range of ``flat_grad`` covering every parameter whose key starts with one of
        ``prefixes`` (parameters of one stage are contiguous in the flat buffer)."""
        rng = [(o, o + n) for k, (o, n) in self._slices.items() if any(k.startswith(p) for p in prefixes)]
        if not rng:
            raise KeyError(prefixes)
        return min(a for a, _ in rng), max(b for _, b in rng)


# ================================================================================================
# Generator
# ================================================================================================
class GeneratorModel(_Link):
    """Drop-in for srgan_train.GeneratorModel (srgan_train.py:421-576).

    >>> model = GeneratorModel()                                      # doctest: +SKIP
    >>> model.forward(x=X, w1=W1, w2=W2, w3=W3).shape               # doctest: +SKIP
    (1, 1, 36, 36)
    >>> model.count_params()                                          # doctest: +SKIP
    8907749
    """

    def __init__(self, inblock_class=None, resblock_class=None, num_residual_blocks: int = 12,
                 residual_scaling: float = 0.1, out_channels: int = 1, *, inter_channels: int = 32,
                 precision: str = "bf16", train_precision: Optional[str] = None, seed: int = 0,
                 init_scale: float = 0.1):
        if precision not in ("bf16", "bf16x3", "fp32"):
            raise ValueError("precision must be 'bf16', 'bf16x3' or 'fp32'")
        if train_precision is None:
            train_precision = "fp32" if precision == "fp32" else "bf16"
        if train_precision not in ("bf16", "fp32"):
            raise ValueError("train_precision must be 'bf16' or 'fp32'")
        if inter_channels not in (32, 64):
            raise ValueError("inter_channels must be 32 or 64 (reference search space, srgan_train.py:283-284)")
        self.num_residual_blocks = int(num_residual_blocks)
        self.residual_scaling = float(residual_scaling)
        self.out_channels = int(out_channels)
        self.inter_channels = int(inter_channels)
        self.precision = precision
        self.train_precision = train_precision
        self._flat = {}
        self._head_images, self._head_tc, self._head_packed_version, self._head_pack_table = None, {}, -1, None
        shapes = layout.generator_shapes(self.num_residual_blocks, self.inter_channels, self.out_channels)
        super().__init__(shapes, layout.init_values(shapes, seed, init_scale))
        self._packed_version = -1
        self._packed = {}
        self._pack_plan = None
        self._pack_gen = 0   # bumps when the packed buffers are (re)allocated: cached pointer tables key on it
        self._ws = {}
        self.persistent_trunk = True   # one-launch trunk kernel (False: one launch per layer, for A/B tests)
        self.paired_trunk = True       # dense-block layer pairing inside the persistent kernel
        self.paired_convs = (1, 3)     # which pairs (conv_k, conv_k+1) are fused: (1, 3) both, (3,) the second only
        self.per_layer_ck16 = False    # per-layer launches in the trunk kernel's 16-channel chunks (bit-exact A/B)
        self.local_trunk = True        # tiles of <= 128 padded positions: image-resident trunk kernel (umma_local.cu)
        # output layer's tap projection inside the first deformable layer's epilogue: bit-identical, but measured
        # SLOWER (the four epilogue warps become the bottleneck: 2.11 -> 2.57 ms to save a 0.25 ms kernel) -> off
        self.fuse_out_projection = False
        # conv_on_W1 (k30 s10) as a split-bf16 tcgen05 GEMM over the 10x10 space-to-depth (False: fp32 CUDA cores)
        self.stem_w1_tensor_core = True
        # tiled tensor-core inference through the model-level C entry points (dbm_gen_forward, csrc/gen_api.cu): the
        # pass / pack tables and the workspace layout are built in C++; False (or any A/B switch above off its
        # default): the same kernels composed call by call from this file
        self.c_model_api = True
        self._cgen, self._cgen_version, self._cgen_ws = None, -1, {}
        # training forward of the first deformable layer as one fused tcgen05 kernel (False: sampler + bf16 GEMM, cols kept)
        self.fused_deform_forward = True
        # its backward re-samples the weight-gradient operand from the forward's bf16 slab8 input with 16-byte gathers
        # (False: from the fp32 NCHW tensor, one 4-byte gather per channel and corner)
        self.resample_from_slab8 = True
        # upper bound of the persistent grid of the trunk's batched weight-gradient launch (0 = every SM but the
        # reserve): in the training step the discriminator's weight gradients run beside it and end the step
        self.trunk_wgrad_ctas = 0
        self._ctx = None

    # ---- serialisation (chainer.serializers.load_npz / save_npz, App. C layout) ----
    def load_npz(self, file, strict: bool = True):
        npz_io.load_npz(file, self, strict=strict)
        return self

    def save_npz(self, file, compression: bool = True):
        npz_io.save_npz(file, self, compression=compression)

    # ---- forward ----
    def __call__(self, x, w1, w2, w3):
        return self.forward(x, w1, w2, w3)

    def forward(self, x, w1, w2, w3) -> Variable:
        """Inference forward: inputs (N,1,h,w), (N,1,10h,10w), (N,2,2h,2w), (N,1,h,w) float32
        (NumPy or torch, host or device) -> Variable with .array (N,1,4(h-2),4(w-2)) on the GPU."""
        x, w1, w2, w3 = (as_device(a) for a in (x, w1, w2, w3))
        self._check_shapes(x, w1, w2, w3)
        if self.precision == "bf16":
            y = self._forward_bf16(x, w1, w2, w3)
        elif self.precision == "bf16x3":
            y = self._forward_split(x, w1, w2, w3)
        else:
            y = self._forward_fp32(x, w1, w2, w3, save=False)
        return Variable(y)

    def forward_train(self, x, w1, w2, w3) -> Variable:
        """Forward that keeps the activations needed by ``backward`` (the reference's graph-building
        forward, srgan_train.py:1222-1227). Stem, upsample and deformable layers run in fp32; the trunk
        (98 % of the trunk+stem FLOPs) runs on the tensor cores when ``train_precision == "bf16"``
        (flat.py / csrc/umma_flat.cu) and in fp32 otherwise."""
        x, w1, w2, w3 = (as_device(a) for a in (x, w1, w2, w3))
        self._check_shapes(x, w1, w2, w3)
        y = self._forward_fp32(x, w1, w2, w3, save=True)
        # lets the generator step pick up the graph the discriminator step built from the same batch
        # (train.train_eval_discriminator(share_generator_forward=True)); the context keeps the inputs alive,
        # so equal pointers + equal in-place version counters + equal weight version identify the same forward
        self._ctx["y"] = y
        self._ctx["key"] = self._forward_key(x, w1, w2, w3)
        return Variable(y)

    def _forward_key(self, x, w1, w2, w3):
        """Identity of a forward: weight version + for every input its address, shape and torch's in-place version
        counter -- an in-place refresh of an input buffer (``copy_``, ``+=`` ...) between the two step functions bumps
        the counter, so stale activations are never reused for new data."""
        return (self.version,) + tuple((t.data_ptr(), tuple(t.shape), t._version) for t in (x, w1, w2, w3))

    def shared_forward(self, x, w1, w2, w3) -> Optional[torch.Tensor]:
        """Output of a preceding ``forward_train`` on exactly these device tensors with the current weights
        (its saved activations are still in place for ``backward``), else None."""
        c = self._ctx
        if c is None or "key" not in c or not all(isinstance(t, torch.Tensor) and t.is_cuda for t in (x, w1, w2, w3)):
            return None
        return c["y"] if self._forward_key(x, w1, w2, w3) == c["key"] else None

    @staticmethod
    def _check_shapes(x, w1, w2, w3):
        if x.dim() != 4 or w1.dim() != 4 or w2.dim() != 4 or w3.dim() != 4:
            raise ValueError("inputs must be 4-D (N, C, H, W) arrays")
        n, c, h, w = x.shape
        ok = (c == 1 and tuple(w1.shape) == (n, 1, 10 * h, 10 * w) and tuple(w2.shape) == (n, 2, 2 * h, 2 * w)
              and tuple(w3.shape) == (n, 1, h, w) and h >= 3 and w >= 3)
        if not ok:
            # Chainer raises InvalidType from F.concat for inconsistent input sizes (srgan_train.py:265)
            raise ValueError(f"inconsistent input shapes: x{tuple(x.shape)} w1{tuple(w1.shape)} "
                             f"w2{tuple(w2.shape)} w3{tuple(w3.shape)}; need w1 = 10x, w2 = 2x (2 ch), w3 = 1x of x")

    def _rdb_prefix(self, i, r):
        return f"residual_network/{i}/residual_dense_block{r}"

    # ---------------- fp32 path ----------------
    def _stem_fp32(self, x, w1, w2, w3, out, c0=0):
        P = self.p
        ops.conv2d_fwd(x, 0, 1, P["input_block/conv_on_X/W"], P["input_block/conv_on_X/b"], out, c0 + 0, 3, 1, 0)
        ops.conv2d_fwd(w1, 0, 1, P["input_block/conv_on_W1/W"], P["input_block/conv_on_W1/b"], out, c0 + 32, 30, 10, 0)
        ops.conv2d_fwd(w2, 0, 2, P["input_block/conv_on_W2/W"], P["input_block/conv_on_W2/b"], out, c0 + 64, 6, 2, 0)
        ops.conv2d_fwd(w3, 0, 1, P["input_block/conv_on_W3/W"], P["input_block/conv_on_W3/b"], out, c0 + 96, 3, 1, 0)

    def _forward_fp32(self, x, w1, w2, w3, save: bool):
        P = self.p
        g = self.inter_channels
        cc = 64 + 4 * g
        beta = self.residual_scaling
        n, _, h, w = x.shape
        H, W = h - 2, w - 2
        a0 = ops.empty(n, 128, H, W)
        self._stem_fp32(x, w1, w2, w3, a0)
        nrdb = 3 * self.num_residual_blocks
        if save and self.train_precision == "bf16":
            ft = self._flat_trunk(n, H, W)
            a3 = ft.forward(a0)
            return self._head_fp32(a3, dict(x=x, w1=w1, w2=w2, w3=w3, a0=a0, flat=ft, H=H, W=W, n=n), save)
        cats = [ops.empty(n, cc, H, W) for _ in range(nrdb + 1)]  # cats[j][:, :64] = input of RDB j
        ops.conv2d_fwd(a0, 0, 128, P["pre_residual_conv_layer/W"], P["pre_residual_conv_layer/b"], cats[0], 0, 3, 1, 1,
                       act=True)
        t5s = []
        j = 0
        for i in range(self.num_residual_blocks):
            rrdb_in = cats[j]
            for r in (1, 2, 3):
                cat = cats[j]
                pre = self._rdb_prefix(i, r)
                for k in (1, 2, 3, 4):
                    cin = 64 + (k - 1) * g
                    ops.conv2d_fwd(cat, 0, cin, P[f"{pre}/conv_layer{k}/W"], P[f"{pre}/conv_layer{k}/b"], cat, cin, 3, 1,
                                   1, act=True)
                t5 = ops.empty(n, 64, H, W)
                ops.conv2d_fwd(cat, 0, cc, P[f"{pre}/conv_layer5/W"], P[f"{pre}/conv_layer5/b"], t5, 0, 3, 1, 1)
                nxt = cats[j + 1]
                # a6 = a5 * beta + a0 (srgan_train.py:358)
                ops.axpby(t5, 0, cat, 0, nxt, 0, 64, beta, 1.0)
                if r == 3:  # a4 = a3 * beta + x (srgan_train.py:402)
                    ops.axpby(nxt, 0, rrdb_in, 0, nxt, 0, 64, beta, 1.0)
                j += 1
        last = cats[nrdb]
        t = ops.empty(n, 64, H, W)
        ops.conv2d_fwd(last, 0, 64, P["post_residual_conv_layer/W"], P["post_residual_conv_layer/b"], t, 0, 3, 1, 1)
        a3 = ops.empty(n, 64, H, W)
        ops.axpby(t, 0, cats[0], 0, a3, 0, 64, 1.0, 1.0)  # a3 = a1 + conv (srgan_train.py:551)
        return self._head_fp32(a3, dict(x=x, w1=w1, w2=w2, w3=w3, a0=a0, cats=cats, H=H, W=W, n=n), save)

    def _flat_trunk(self, n, H, W):
        from . import flat
        pk = self._pack(self.PACK_TRAIN_LOCAL if (flat.local_trunk_fits(H, W) and self.inter_channels == 32)
                        else self.PACK_TRAIN_CHAIN)
        ft = self._flat.get((n, H, W))
        if ft is None:
            ft = self._flat[(n, H, W)] = flat.FlatTrunk(self, n, H, W)
        ft.build(pk)
        return ft

    def _head_fp32(self, a3, ctx, save: bool):
        """Upsample convs + the two deformable layers (srgan_train.py:553-574), fp32."""
        P = self.p
        n, H, W = ctx["n"], ctx["H"], ctx["W"]
        tc = self._head_convs(n, H, W) if (save and self.train_precision == "bf16") else None

        def conv(key, x, act):
            if tc is not None:   # tcgen05 (flat.FlatConv): bf16 operands, fp32 accumulation, bias (+ LeakyReLU) fused
                return tc[key].forward(x)
            w = P[f"{key}/W"]
            out = ops.empty(n, w.shape[0], x.shape[2], x.shape[3])
            ops.conv2d_fwd(x, 0, 64, w, P[f"{key}/b"], out, 0, 3, 1, 1, act=act)
            return out

        u1 = ops.upsample2_fwd(a3)
        c1 = conv("post_upsample_conv_layer_1", u1, True)
        u2 = ops.upsample2_fwd(c1)
        c2 = conv("post_upsample_conv_layer_2", u2, True)
        off1 = conv("final_conv_layer1/offset_conv", c2, False)
        if tc is not None and self.fused_deform_forward:
            # gather + tcgen05 contraction + bias + LeakyReLU in one kernel; backward re-samples (no 382 MB cols buffer
            # on the forward's critical path)
            wq, _ = self._packed["final_conv_layer1/deform_conv"]
            d1, c2_slab8 = ops.deform_conv_fwd_fused(c2, off1, wq, P["final_conv_layer1/deform_conv/b"], act=True,
                                                     keep_slab8=True)
            cols1 = None
            if save:
                ctx["c2_slab8"] = c2_slab8   # backward re-samples from the very operand the forward gathered from
        else:
            d1, cols1 = ops.deform_conv_fwd(c2, off1, P["final_conv_layer1/deform_conv/W"],
                                            P["final_conv_layer1/deform_conv/b"], act=True, tc=tc is not None)
        off2 = conv("final_conv_layer2/offset_conv", d1, False)
        if self.out_channels == 1:   # tap projection: 9 projected planes instead of a 576-row cols buffer
            y, cols2 = ops.deform1_conv_fwd(d1, off2, P["final_conv_layer2/deform_conv/W"],
                                            P["final_conv_layer2/deform_conv/b"])
        else:
            y, cols2 = ops.deform_conv_fwd(d1, off2, P["final_conv_layer2/deform_conv/W"],
                                           P["final_conv_layer2/deform_conv/b"], act=False)
        if save:
            ctx.update(u1=u1, c1=c1, u2=u2, c2=c2, off1=off1, d1=d1, cols1=cols1, off2=off2, cols2=cols2, head_tc=tc)
            self._ctx = ctx
        return y

    HEAD_TC_KEYS = ("post_upsample_conv_layer_1", "post_upsample_conv_layer_2", "final_conv_layer1/offset_conv",
                    "final_conv_layer2/offset_conv")

    def _head_convs(self, n, H, W):
        """flat.FlatConv objects of the four plain 3x3 convolutions of the head for this batch shape; their
        operand images are re-packed (one launch) whenever the weights changed."""
        from . import flat
        if self._head_images is None:
            self._head_images = {k: flat.ConvImages(self.p[f"{k}/W"], self.p[f"{k}/b"]) for k in self.HEAD_TC_KEYS}
        if self._head_packed_version != self.version:
            self._head_pack_table = flat.pack_images(list(self._head_images.values()), self._head_pack_table)
            self._head_packed_version = self.version
        tc = self._head_tc.get((n, H, W))
        if tc is None:
            sizes = {"post_upsample_conv_layer_1": 2, "post_upsample_conv_layer_2": 4,
                     "final_conv_layer1/offset_conv": 4, "final_conv_layer2/offset_conv": 4}
            tc = {k: flat.FlatConv(self._head_images[k], self.g[f"{k}/W"], n, sizes[k] * H, sizes[k] * W,
                                   act=k.startswith("post_upsample")) for k in self.HEAD_TC_KEYS}
            self._head_tc[(n, H, W)] = tc
        return tc

    def backward(self, dy: torch.Tensor, on_ready=None):
        """Accumulates d(loss)/d(params) into ``flat_grad`` given d(loss)/d(output) (N,1,4H,4W);
        replaces g_loss.backward() for the generator (srgan_train.py:1256). No gradient wrt the
        inputs is produced (no caller needs it). ``on_ready(lo, hi)`` is called as soon as the
        gradients of flat_grad[lo:hi] are final, on the stream that produced them, so a data-parallel caller can
        all-reduce that bucket while the rest of backward runs: tensor-core path = three buckets (head, whole trunk,
        stem; see below), fp32 path = head, then each RRDB from last to first, then the stem."""
        if self._ctx is None:
            raise RuntimeError("backward() needs a preceding forward_train()")
        ready = (lambda *pre: on_ready(*self.grad_range(pre))) if on_ready is not None else (lambda *pre: None)
        c = self._ctx
        P, G = self.p, self.g
        g = self.inter_channels
        cc = 64 + 4 * g
        beta = self.residual_scaling
        n, H, W = c["n"], c["H"], c["W"]
        dy = dy.contiguous()
        # ---- final_conv_layer2 (deformable, no activation) ----
        tc = c.get("head_tc")

        def conv_bwd(key, x, dz, dx_accumulate_into=None):
            """dW, db of a plain 3x3 conv of the head and its data gradient (added to ``dx_accumulate_into``
            or returned)."""
            if tc is not None:
                aux = ops._aux_stream()
                aux.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(aux):   # bias / weight gradients beside the data-gradient chain
                    ops.call("dbm_bias_grad_f32", dz.data_ptr(), dz.shape[1] * dz.shape[2] * dz.shape[3],
                             G[f"{key}/b"].data_ptr(), n, dz.shape[1], dz.shape[2] * dz.shape[3], ops.stream())
                dx = tc[key].backward(dz, wgrad_stream=aux)
                if dx_accumulate_into is None:
                    return dx
                ops.axpby(dx, 0, dx_accumulate_into, 0, dx_accumulate_into, 0, 64, 1.0, 1.0)
                return dx_accumulate_into
            ops.conv2d_bwd_weight(x, 0, 64, dz, 0, G[f"{key}/W"], 3, 1, 1, db=G[f"{key}/b"])
            if dx_accumulate_into is not None:
                ops.conv2d_bwd_data(dz, 0, P[f"{key}/W"], dx_accumulate_into, 0, 64, 3, 1, 1, accumulate=True)
                return dx_accumulate_into
            dx = ops.empty(*x.shape)
            ops.conv2d_bwd_data(dz, 0, P[f"{key}/W"], dx, 0, 64, 3, 1, 1)
            return dx

        if self.out_channels == 1:
            dd1 = ops.empty(n, 64, 4 * H, 4 * W)
            doff2 = ops.deform1_conv_bwd(c["d1"], c["off2"], P["final_conv_layer2/deform_conv/W"], c["cols2"], dy,
                                         G["final_conv_layer2/deform_conv/W"], G["final_conv_layer2/deform_conv/b"], dd1)
        else:
            dd1 = ops.zeros(n, 64, 4 * H, 4 * W)
            doff2 = ops.deform_conv_bwd(c["d1"], c["off2"], P["final_conv_layer2/deform_conv/W"], c["cols2"], dy,
                                        G["final_conv_layer2/deform_conv/W"], G["final_conv_layer2/deform_conv/b"], dd1)
        conv_bwd("final_conv_layer2/offset_conv", c["d1"], doff2, dx_accumulate_into=dd1)
        ops.lrelu_bwd(dd1, 0, c["d1"], 0, dd1, 0, 64)
        # ---- final_conv_layer1 ----
        dc2 = ops.zeros(n, 64, 4 * H, 4 * W)
        if c["cols1"] is not None:
            cols1 = c["cols1"]
        elif c.get("c2_slab8") is not None and self.resample_from_slab8:
            cols1 = ops.deform_sample_slab8(c["c2_slab8"], c["off1"])
        else:
            cols1 = ops.deform_sample(c["c2"], c["off1"])
        doff1 = ops.deform_conv_bwd(c["c2"], c["off1"], P["final_conv_layer1/deform_conv/W"], cols1, dd1,
                                    G["final_conv_layer1/deform_conv/W"], G["final_conv_layer1/deform_conv/b"], dc2,
                                    tc=c.get("head_tc") is not None)
        conv_bwd("final_conv_layer1/offset_conv", c["c2"], doff1, dx_accumulate_into=dc2)
        del dd1, doff1, doff2
        # ---- upsample convs ----
        ops.lrelu_bwd(dc2, 0, c["c2"], 0, dc2, 0, 64)
        du2 = conv_bwd("post_upsample_conv_layer_2", c["u2"], dc2)
        dc1 = ops.upsample2_bwd(du2)
        del du2, dc2
        ops.lrelu_bwd(dc1, 0, c["c1"], 0, dc1, 0, 64)
        du1 = conv_bwd("post_upsample_conv_layer_1", c["u1"], dc1)
        da3 = ops.upsample2_bwd(du1)  # = d a1 (skip) = d (post-res conv output)
        del du1, dc1
        if "flat" in c:
            # tensor-core trunk: data-gradient chain, batched weight/bias gradients (flat.py).
            # Three gradient buckets, each handed on the moment it is final so that a data-parallel caller's
            # all-reduce (GradBucketReducer: the comm stream waits for the stream current at the hand-over) runs
            # under what is still to come:
            #   head  (upsample + deformable layers): its weight / bias gradients were launched on ``aux`` beside the
            #         data-gradient chain; handed over on that stream, reduced under the whole trunk backward;
            #   trunk (pre-residual conv .. post-residual conv): one batched launch + reduction on the side stream
            #         ``aux`` beside the stem's backward, handed over ON that stream;
            #   stem  (input_block): after the stem's weight gradients on the main stream.
            cur, aux = torch.cuda.current_stream(), ops._aux_stream()
            with torch.cuda.stream(aux):
                ready("post_upsample_conv_layer", "final_conv_layer")
            da0 = c["flat"].backward(da3, wgrad_stream=aux)
            with torch.cuda.stream(aux):
                ready("pre_residual_conv_layer", "residual_network/", "post_residual_conv_layer")
            self._stem_bwd(c, da0, lambda *pre: None)
            ready("input_block/")
            cur.wait_stream(aux)
            return
        # ---- post-residual conv ----
        cats = c["cats"]
        nrdb = 3 * self.num_residual_blocks
        ops.conv2d_bwd_weight(cats[nrdb], 0, 64, da3, 0, G["post_residual_conv_layer/W"], 3, 1, 1,
                              db=G["post_residual_conv_layer/b"])
        dcur = ops.empty(n, 64, H, W)  # gradient wrt the trunk output
        ops.conv2d_bwd_data(da3, 0, P["post_residual_conv_layer/W"], dcur, 0, 64, 3, 1, 1)
        ready("post_residual_conv_layer", "post_upsample_conv_layer", "final_conv_layer")
        # ---- trunk, reversed ----
        j = nrdb
        for i in reversed(range(self.num_residual_blocks)):
            d_rrdb_out = dcur  # out = x + beta * a3
            d_rdb_out = ops.empty(n, 64, H, W)
            ops.axpby(d_rrdb_out, 0, None, 0, d_rdb_out, 0, 64, beta, 0.0)
            for r in (3, 2, 1):
                j -= 1
                cat = cats[j]
                pre = self._rdb_prefix(i, r)
                # a6 = a0 + beta * a5
                d5 = ops.empty(n, 64, H, W)
                ops.axpby(d_rdb_out, 0, None, 0, d5, 0, 64, beta, 0.0)
                ops.conv2d_bwd_weight(cat, 0, cc, d5, 0, G[f"{pre}/conv_layer5/W"], 3, 1, 1, db=G[f"{pre}/conv_layer5/b"])
                dcat = ops.empty(n, cc, H, W)
                ops.conv2d_bwd_data(d5, 0, P[f"{pre}/conv_layer5/W"], dcat, 0, cc, 3, 1, 1)
                ops.axpby(dcat, 0, d_rdb_out, 0, dcat, 0, 64, 1.0, 1.0)  # + d a0 (skip)
                for k in (4, 3, 2, 1):
                    cin = 64 + (k - 1) * g
                    ops.lrelu_bwd(dcat, cin, cat, cin, dcat, cin, g)
                    ops.conv2d_bwd_weight(cat, 0, cin, dcat, cin, G[f"{pre}/conv_layer{k}/W"], 3, 1, 1,
                                          db=G[f"{pre}/conv_layer{k}/b"])
                    ops.conv2d_bwd_data(dcat, cin, P[f"{pre}/conv_layer{k}/W"], dcat, 0, cin, 3, 1, 1, accumulate=True)
                d_rdb_out = ops.empty(n, 64, H, W)
                ops.axpby(dcat, 0, None, 0, d_rdb_out, 0, 64, 1.0, 0.0)
            # RRDB skip: d x += d out
            dcur = ops.empty(n, 64, H, W)
            ops.axpby(d_rdb_out, 0, d_rrdb_out, 0, dcur, 0, 64, 1.0, 1.0)
            ready(f"residual_network/{i}/")
        # ---- a1 = lrelu(pre_res(a0)); total gradient = trunk input + skip to a3 ----
        da1 = ops.empty(n, 64, H, W)
        ops.axpby(dcur, 0, da3, 0, da1, 0, 64, 1.0, 1.0)
        ops.lrelu_bwd(da1, 0, cats[0], 0, da1, 0, 64)
        ops.conv2d_bwd_weight(c["a0"], 0, 128, da1, 0, G["pre_residual_conv_layer/W"], 3, 1, 1,
                              db=G["pre_residual_conv_layer/b"])
        da0 = ops.empty(n, 128, H, W)
        ops.conv2d_bwd_data(da1, 0, P["pre_residual_conv_layer/W"], da0, 0, 128, 3, 1, 1)
        self._stem_bwd(c, da0, ready)

    def _stem_bwd(self, c, da0, ready):
        G = self.g
        # ---- stem weights ----
        ops.conv2d_bwd_weight(c["x"], 0, 1, da0, 0, G["input_block/conv_on_X/W"], 3, 1, 0, db=G["input_block/conv_on_X/b"])
        ops.conv2d_bwd_weight(c["w1"], 0, 1, da0, 32, G["input_block/conv_on_W1/W"], 30, 10, 0,
                              db=G["input_block/conv_on_W1/b"])
        ops.conv2d_bwd_weight(c["w2"], 0, 2, da0, 64, G["input_block/conv_on_W2/W"], 6, 2, 0,
                              db=G["input_block/conv_on_W2/b"])
        ops.conv2d_bwd_weight(c["w3"], 0, 1, da0, 96, G["input_block/conv_on_W3/W"], 3, 1, 0,
                              db=G["input_block/conv_on_W3/b"])
        ready("input_block/", "pre_residual_conv_layer")
        self._ctx = None

    # ---------------- bf16 tensor-core path (inference) ----------------
    # groups of packed operand images (a training step must not pay for the inference-only ones)
    PACK_INFER = ("io", "trunk16", "infer", "deform")                 # tiled / persistent tensor-core inference
    PACK_INFER_LOCAL = ("io", "stat", "infer", "deform")              # inference on tiles that fit the image-resident kernel
    PACK_TRAIN_LOCAL = ("io", "stat", "dgrad", "deform")              # training, image-resident trunk
    PACK_TRAIN_CHAIN = ("io", "trunk16", "stat", "dgrad", "deform")   # training, flat chain (any tile size)
    PACK_SPLIT = ("split",)                                           # precision="bf16x3": split-bf16 trunk + upsample convs

    def _pack(self, groups=None):
        """bf16 UMMA operand images of every 3x3 filter (+ the stem's tap-major fp32 filters). The
        buffers and device tables describing them are created once; after a weight update (training)
        the groups a caller needs are refreshed by one table-driven launch each (dbm_pack_conv3x3_table):
          io      pre-/post-residual conv in 16-channel chunks (every trunk kernel)
          trunk16 dense-block convs in 16-channel chunks (persistent inference trunk, flat training chain)
          infer   32-channel-chunk images, pair/tail images, head convs, stem filters, padded biases
          stat    input-stationary slices (image-resident small-tile trunk)
          dgrad   transposed + flipped filters (data gradients)
          deform  the first deformable layer's 64-channel-chunk image (inference and the fused training forward)"""
        if groups is None:
            groups = self.PACK_INFER
        P = self.p
        if self._pack_plan is None:
            pk = {}
            entries = {g: [] for g in ("io", "trunk16", "infer", "stat", "dgrad", "deform", "split")}
            pad_biases = []   # (padded bias buffer, source bias)

            def image(cin, cout_padded):
                return ops.zeros(9 * cin * cout_padded, dtype=torch.bfloat16)

            def entry(grp, w, out, o, o0, cin, cin_total, c0, coutp, ck, mode=0):
                entries[grp].append((w.data_ptr(), out.data_ptr(), o, o0, cin, cin_total, c0, coutp, ck, mode))

            def add(key, cout_padded, trunk=None, ck=32, grp="infer"):
                w, b = P[f"{key}/W"], P[f"{key}/b"]
                o, cin = w.shape[0], w.shape[1]
                if b.numel() < cout_padded:
                    bp = ops.zeros(cout_padded)
                    pad_biases.append((bp, b))
                else:
                    bp = b
                img = image(cin, cout_padded)
                entry(grp, w, img, o, 0, cin, cin, 0, cout_padded, ck)
                pk[key] = (img, bp)
                if trunk is not None:
                    # the trunk kernels stream every layer in 16-channel chunks
                    img16 = image(cin, cout_padded)
                    entry(trunk, w, img16, o, 0, cin, cin, 0, cout_padded, 16)
                    pk[key + "@trunk"] = (img16, bp)
                    if self.train_precision == "bf16":
                        # data-gradient operand (transposed + flipped filter): GEMM N = cin, K = cout; the flat kernels
                        # take N <= 192, so wider filters (inter_channels = 64: conv4 256, conv5 320) are packed as
                        # N-slices, one launch each
                        slices = []
                        for c0 in range(0, cin, 192):
                            wdt = min(192, cin - c0)
                            imgd = image(wdt, o)
                            entry("dgrad", w, imgd, wdt, 0, o, cin, c0, wdt, 16, mode=1)
                            slices.append((c0, wdt, imgd))
                        if len(slices) == 1:
                            pk[key + "@dgrad"] = slices[0][2]
                        pk[key + "@dgrad_slices"] = slices

            def add_sliced(grp, name, slices, cin, coutp, bias, elems=1, mode=0):
                # one image assembled from filter slices (wkey, O, o0, cin_total, c0); elems = 3 for split-bf16
                img = ops.zeros(elems * 9 * cin * coutp, dtype=torch.bfloat16)
                for wkey, o, o0, cin_total, c0 in slices:
                    entry(grp, P[wkey], img, o, o0, cin, cin_total, c0, coutp, 16, mode)
                pk[name] = (img, P[bias])

            def pair_images(pre):
                # dense-block pairing (layout.trunk_plan, inter_channels = 32): the head image pair{k} holds conv_k and
                # the rows of conv_{k+1} over their shared inputs (one 64-wide MMA pass), the tail image tail{k+1}
                # conv_{k+1}'s rows over a_k. (name, slices, cin, coutp, bias key) per image.
                out = []
                for k in (1, 3):
                    cin = 64 + (k - 1) * 32
                    wa, wb = f"{pre}/conv_layer{k}/W", f"{pre}/conv_layer{k + 1}/W"
                    out.append((f"{pre}/pair{k}", [(wa, 32, 0, cin, 0), (wb, 32, 32, cin + 32, 0)], cin, 64,
                                f"{pre}/conv_layer{k}/b"))
                    out.append((f"{pre}/tail{k + 1}", [(wb, 32, 0, cin + 32, cin)], 32, 32, f"{pre}/conv_layer{k + 1}/b"))
                return out

            add("pre_residual_conv_layer", 64, trunk="io")
            for i in range(self.num_residual_blocks):
                for r in (1, 2, 3):
                    pre = self._rdb_prefix(i, r)
                    for k in (1, 2, 3, 4):
                        add(f"{pre}/conv_layer{k}", self.inter_channels, trunk="trunk16")
                    add(f"{pre}/conv_layer5", 64, trunk="trunk16")
            add("post_residual_conv_layer", 64, trunk="io")
            if self.inter_channels == 32:
                for i in range(self.num_residual_blocks):
                    for r in (1, 2, 3):
                        for name, slices, cin, coutp, bias in pair_images(self._rdb_prefix(i, r)):
                            add_sliced("infer", name, slices, cin, coutp, bias)
                # input-stationary slices for the image-resident small-tile trunk (csrc/umma_local.cu): pass s
                # contracts block a_s (a0 = 64 channels, a1..a4 = 32) against its rows in conv_{s+1}..conv_5
                # stacked along N = 192 - 32 s
                for i in range(self.num_residual_blocks):
                    for r in (1, 2, 3):
                        pre = self._rdb_prefix(i, r)
                        for s_ in range(5):
                            cblk, c0 = (64, 0) if s_ == 0 else (32, 64 + 32 * (s_ - 1))
                            ncol = 192 - 32 * s_
                            stat = image(cblk, ncol)
                            for k in range(s_ + 1, 6):
                                entry("stat", P[f"{pre}/conv_layer{k}/W"], stat, 64 if k == 5 else 32, 32 * (k - 1 - s_),
                                      cblk, 64 + 32 * (k - 1), c0, ncol, 16)
                            pk[f"{pre}/stat{s_}"] = stat
            if self.precision == "bf16x3":
                # split-bf16 operand images (dbm_trunk_umma_split): per 16-channel chunk [w_hi | w_hi | w_lo], 3x the
                # size of a bf16 image; the trunk's passes (paired plan for inter_channels = 32) and the upsample convs
                def add_split(name, slices, cin, coutp, bias):
                    add_sliced("split", name + "@split", slices, cin, coutp, bias, elems=3, mode=16)

                g_ = self.inter_channels
                for key in ("pre_residual_conv_layer", "post_residual_conv_layer", "post_upsample_conv_layer_1",
                            "post_upsample_conv_layer_2"):
                    w = P[f"{key}/W"]
                    add_split(key, [(f"{key}/W", w.shape[0], 0, w.shape[1], 0)], w.shape[1], 64, f"{key}/b")
                for i in range(self.num_residual_blocks):
                    for r in (1, 2, 3):
                        pre = self._rdb_prefix(i, r)
                        add_split(f"{pre}/conv_layer5", [(f"{pre}/conv_layer5/W", 64, 0, 64 + 4 * g_, 0)], 64 + 4 * g_, 64,
                                  f"{pre}/conv_layer5/b")
                        if g_ == 32:
                            for name, slices, cin, coutp, bias in pair_images(pre):
                                add_split(name, slices, cin, coutp, bias)
                        else:
                            for k in (1, 2, 3, 4):
                                cin = 64 + (k - 1) * g_
                                add_split(f"{pre}/conv_layer{k}", [(f"{pre}/conv_layer{k}/W", g_, 0, cin, 0)], cin, g_,
                                          f"{pre}/conv_layer{k}/b")
            for key in ("post_upsample_conv_layer_1", "post_upsample_conv_layer_2"):
                add(key, 64)
            add("final_conv_layer1/offset_conv", 32)
            add("final_conv_layer2/offset_conv", 32)
            add("final_conv_layer1/deform_conv", 64, ck=64, grp="deform")
            # stem filters, tap-major, and the concatenated stem bias
            taps = {k: int(P[f"input_block/conv_on_{k}/W"][0].numel()) for k in ("X", "W1", "W2", "W3")}
            pk["stem"] = (ops.empty(taps["W1"], 32), ops.empty(taps["X"] + taps["W2"] + taps["W3"], 32), ops.empty(128))
            # conv_on_W1 on the tensor cores (3x3 valid conv over the 10x10 space-to-depth, split-bf16 operands)
            pk["stem_w1_tc"] = ops.empty(9 * 320 * 32, dtype=torch.bfloat16)
            tables = {}
            for g, ent in entries.items():
                if ent:
                    table = np.array(ent, dtype=PACK_ENTRY_DTYPE)
                    tables[g] = dict(table=torch.from_numpy(table.view(np.uint8).copy()).cuda(), n=len(ent),
                                     max_elements=max(9 * e[4] * e[7] for e in ent))
            self._pack_plan = dict(tables=tables, pad_biases=pad_biases, taps=taps)
            self._packed = pk
            self._pack_versions = {g: -1 for g in tables}
            self._pack_gen += 1
        plan, pk = self._pack_plan, self._packed
        for g in groups:
            t = plan["tables"].get(g)
            if t is None or self._pack_versions[g] == self.version:
                continue
            ops.call("dbm_pack_conv3x3_table", t["table"].data_ptr(), t["n"], t["max_elements"], ops.stream())
            if g == "infer":
                for bp, b in plan["pad_biases"]:
                    ops.axpby(b.view(1, b.numel(), 1, 1), 0, None, 0, bp.view(1, bp.numel(), 1, 1), 0, b.numel(), 1.0, 0.0)
                wt1, wts, bias128 = pk["stem"]
                r0 = 0
                for k, dst in (("W1", wt1), ("X", wts), ("W2", wts), ("W3", wts)):
                    nt = plan["taps"][k]
                    row = 0 if k == "W1" else r0
                    ops.call("dbm_transpose_f32", P[f"input_block/conv_on_{k}/W"].data_ptr(), dst[row:].data_ptr(), 32, nt,
                             ops.stream())
                    if k != "W1":
                        r0 += nt
                for j, k in enumerate(("X", "W1", "W2", "W3")):
                    ops.axpby(P[f"input_block/conv_on_{k}/b"].view(1, 32, 1, 1), 0, None, 0,
                              bias128.view(1, 128, 1, 1), 32 * j, 32, 1.0, 0.0)
                ops.call("dbm_pack_stem_w1", P["input_block/conv_on_W1/W"].data_ptr(), pk["stem_w1_tc"].data_ptr(),
                         ops.stream())
            self._pack_versions[g] = self.version
        return pk

    def _trunk_workspace(self, n, H, W):
        """Per-shape persistent buffers of the trunk + the device layer table of the persistent
        trunk kernel (pointers are baked into the table, so the buffers are cached)."""
        key = (n, H, W)
        ws = self._ws.get(key)
        pk = self._pack()
        if ws is not None and ws["version"] == (self._pack_gen, self.persistent_trunk, self.paired_trunk,
                                                self.per_layer_ck16, self.paired_convs):
            return ws
        bf = torch.bfloat16
        g = self.inter_channels
        ccs = (64 + 4 * g) // 8
        # pairing keeps partial sums in tensor memory between a head and its tail on the same CTA; the schedule's
        # deadlock-freedom argument needs a unit's neighbours (+- one row of 16-pixel-wide units) to lie within one
        # round of CTAs, i.e. images narrower than ~2000 px (csrc/umma_trunk.cu, "schedule")
        paired = self.persistent_trunk and self.paired_trunk and g == 32 and (W + 15) // 16 + 2 <= 128
        if ws is None:
            ws = dict(s0=ops.empty(n, 16, H, W, 8, dtype=bf), cat=[ops.empty(n, ccs, H, W, 8, dtype=bf) for _ in range(2)],
                      a1_f32=ops.empty(n, 16, H, W, 4), f32=[ops.empty(n, 16, H, W, 4) for _ in range(3)],
                      u1=ops.empty(n, 8, 2 * H, 2 * W, 8, dtype=bf))
        plan = layout.trunk_plan(self.num_residual_blocks, g, self.residual_scaling, paired, self.paired_convs)
        # the pair / tail images (modes 1, 2) exist in one form; the persistent kernel (and the per-layer kernel with
        # per_layer_ck16) streams the other filters in 16-channel chunks
        suffix = "@trunk" if self.persistent_trunk or self.per_layer_ck16 else ""
        layers = self._bind_trunk_plan(plan, lambda p: pk[p["image"] + ("" if p["mode"] else suffix)][0], ws, 1)
        table = np.array(layers, dtype=TRUNK_LAYER_DTYPE)
        ws["layers"] = layers
        # executed MMA FLOPs (= algorithmic: pairing moves work, it adds none)
        ws["flops"] = float(sum(2.0 * 9 * p["cin"] * p["cout"] * n * H * W for p in plan))
        ws["table"] = torch.from_numpy(table.view(np.uint8).copy()).cuda()
        tiles = ((H + 31) // 32) * ((W + 15) // 16)   # 32-row x 16-column units (kTH x kTW in umma_trunk.cu)
        ws["flags"] = ops.empty(len(layers) * n * tiles, dtype=torch.int32)
        ws["version"] = (self._pack_gen, self.persistent_trunk, self.paired_trunk, self.per_layer_ck16, self.paired_convs)
        self._ws[key] = ws
        return ws

    def _bind_trunk_plan(self, plan, image, ws, slabs_per_cs):
        """TrunkLayer rows (TRUNK_LAYER_DTYPE) of layout.trunk_plan records: ``image(p)`` is the packed filter image of
        pass p, its buffer names are the workspace's tensors. ``out_cs_total`` counts logical slabs, out.shape[1] //
        ``slabs_per_cs`` (2 for the split path, whose buffers hold a hi and a lo slab per logical slab)."""
        bufs = dict(cat0=ws["cat"][0], cat1=ws["cat"][1], a1=ws["a1_f32"],
                    **{f"f32_{i}": t for i, t in enumerate(ws["f32"])}, **{k: ws[k] for k in ("u1", "u2", "c2f") if k in ws})
        ptr = lambda name: bufs[name].data_ptr() if name is not None else 0
        return [(image(p).data_ptr(), self.p[p["bias"]].data_ptr(), ptr(p["out"]), ptr(p["out_f32"]), ptr(p["res1"]),
                 ptr(p["res2"]), 0, p["cin"], p["cout"], p["in_map"], p["in_cs0"], p["act"], p["up2"],
                 bufs[p["out"]].shape[1] // slabs_per_cs if p["out"] is not None else 0, p["out_cs0"], p["cout_main"], 16,
                 p["beta"], p["mode"], (0,) * 6) for p in plan]

    def _run_trunk(self, ws, n, H, W):
        if self.persistent_trunk:
            ops.call("dbm_trunk_umma", ws["table"].data_ptr(), len(ws["layers"]), n, H, W, ws["s0"].data_ptr(), 16,
                     ws["cat"][0].data_ptr(), ws["cat"][1].data_ptr(), ws["cat"][0].shape[1], ws["flags"].data_ptr(),
                     ops.stream())
            return
        # one launch per layer (kept for A/B measurements of the persistent kernel)
        srcs = (ws["s0"], ws["cat"][0], ws["cat"][1])
        ops.call("dbm_debug_set", 2, int(self.per_layer_ck16))
        for (wq, bq, out, out_f32, res1, res2, _stash, cin, cout, in_map, _cs0, act, up2, out_cs_total, out_cs0, _cm,
             _r1cs, beta_, _mode, _pad) in ws["layers"]:
            inp = srcs[in_map]
            ops.call("dbm_conv3x3_umma", inp.data_ptr(), inp.shape[1], cin, wq, bq, cout, n, H, W, float(beta_), act, up2,
                     out or None, out_cs_total, out_cs0, out_f32 or None, 16, 0, res1 or None, res2 or None, ops.stream())
        ops.call("dbm_debug_set", 2, 0)

    def _local_workspace(self, n, H, W, pk):
        """Buffers + pass table of the image-resident trunk (csrc/umma_local.cu) for inference on small tiles."""
        from . import flat
        key = ("local", n, H, W)
        ws = self._ws.get(key)
        if ws is None or ws["version"] != (self._pack_gen, self.residual_scaling):
            geom = flat.geometry(n, H, W)
            if ws is None:
                ws = dict(s0=torch.zeros(16, geom["Pg"], 8, dtype=torch.bfloat16, device="cuda"),
                          x=torch.empty(2, n * 16 * 128 * 4, dtype=torch.float32, device="cuda"),
                          u1=ops.empty(n, 8, 2 * H, 2 * W, 8, dtype=torch.bfloat16))
            tab = flat.local_forward_table(self, pk, 3 * self.num_residual_blocks, self.residual_scaling,
                                           up2_out=ws["u1"].data_ptr())
            ws["table"] = torch.from_numpy(tab.view(np.uint8).reshape(-1).copy()).cuda()
            ws["count"] = len(tab)
            ws["version"] = (self._pack_gen, self.residual_scaling)
            self._ws[key] = ws
        return ws

    def _c_forward_applies(self):
        return (self.c_model_api and self.persistent_trunk and self.paired_trunk and self.paired_convs == (1, 3)
                and not self.per_layer_ck16
                and self.stem_w1_tensor_core and not self.fuse_out_projection and self.out_channels == 1)

    def _forward_c_api(self, x, w1, w2, w3):
        """GeneratorModel.forward through dbm_gen_forward: this class only owns the flat parameter buffer (bound into
        the handle) and the workspace allocation."""
        import ctypes
        n, _, h, w = x.shape
        if self._cgen is None or self._cgen[1] != self.residual_scaling:
            self._c_release()
            hnd = ctypes.c_void_p()
            ops.call("dbm_gen_create", self.num_residual_blocks, float(self.residual_scaling), self.inter_channels,
                     ctypes.byref(hnd))
            ops.call("dbm_gen_bind_params", hnd, self.flat.data_ptr())
            ops.call("dbm_gen_set_precision", hnd, 1 if self.precision == "bf16x3" else 0)
            self._cgen, self._cgen_version = (hnd, self.residual_scaling), -1
        hnd = self._cgen[0]
        if self._cgen_version != self.version:
            ops.call("dbm_gen_mark_updated", hnd)
            self._cgen_version = self.version
        ws = self._cgen_ws.get((n, h, w))
        if ws is None:
            from . import _lib
            nbytes = int(_lib.load().dbm_gen_workspace_bytes(hnd, n, h, w))
            buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device="cuda")
            ptr = (buf.data_ptr() + 1023) & ~1023
            ws = self._cgen_ws[(n, h, w)] = (buf, ptr, nbytes)
        y = ops.empty(n, 1, 4 * (h - 2), 4 * (w - 2))
        ops.call("dbm_gen_forward", hnd, x.data_ptr(), w1.data_ptr(), w2.data_ptr(), w3.data_ptr(), n, h, w,
                 y.data_ptr(), ws[1], ws[2], ops.stream())
        return y

    def _c_release(self):
        if getattr(self, "_cgen", None) is not None:
            try:
                torch.cuda.synchronize()
                ops.call("dbm_gen_destroy", self._cgen[0])
            except Exception:
                pass
            self._cgen, self._cgen_ws = None, {}

    def __del__(self):
        self._c_release()

    # ---- precision="bf16x3": split-bf16 tensor-core path (fp32-grade results) ----
    def _split_workspace(self, n, H, W, pk):
        """Buffers + pass tables of the split-bf16 path: the trunk table (same passes as the bf16 path, dense-block
        pairing included) and one single-pass table per upsample conv (the same kernel at 2x / 4x the resolution)."""
        key = ("split", n, H, W)
        ws = self._ws.get(key)
        if ws is not None and ws["version"] == (self._pack_gen, self.residual_scaling):
            return ws
        bf = torch.bfloat16
        g = self.inter_channels
        ccs = (64 + 4 * g) // 8
        if ws is None:
            ws = dict(s0=ops.empty(n, 32, H, W, 8, dtype=bf), cat=[ops.empty(n, 2 * ccs, H, W, 8, dtype=bf) for _ in range(2)],
                      a1_f32=ops.empty(n, 16, H, W, 4), f32=[ops.empty(n, 16, H, W, 4) for _ in range(3)],
                      u1=ops.empty(n, 16, 2 * H, 2 * W, 8, dtype=bf), u2=ops.empty(n, 16, 4 * H, 4 * W, 8, dtype=bf),
                      c2f=ops.empty(n, 16, 4 * H, 4 * W, 4))
        paired = g == 32 and (W + 15) // 16 + 2 <= 128
        if g == 32 and not paired:   # only the paired images are packed for the split path
            raise ValueError("precision='bf16x3': tiles wider than ~2000 px are not supported")
        image = lambda p: pk[p["image"] + "@split"][0]
        layers = self._bind_trunk_plan(layout.trunk_plan(self.num_residual_blocks, g, self.residual_scaling, paired),
                                       image, ws, 2)
        up1 = self._bind_trunk_plan([layout.trunk_pass("post_upsample_conv_layer_1", 64, 64, 0, act=1, out="u2", up2=1)],
                                    image, ws, 2)
        up2 = self._bind_trunk_plan([layout.trunk_pass("post_upsample_conv_layer_2", 64, 64, 0, act=1, out_f32="c2f")],
                                    image, ws, 2)
        dev = lambda rows: torch.from_numpy(np.array(rows, dtype=TRUNK_LAYER_DTYPE).view(np.uint8).copy()).cuda()
        units = lambda h_, w_: n * ((h_ + 31) // 32) * ((w_ + 15) // 16)
        ws.update(tables=[dev(layers), dev(up1), dev(up2)], counts=[len(layers), 1, 1],
                  flags=[ops.empty(len(layers) * units(H, W), dtype=torch.int32),
                         ops.empty(units(2 * H, 2 * W), dtype=torch.int32), ops.empty(units(4 * H, 4 * W), dtype=torch.int32)],
                  version=(self._pack_gen, self.residual_scaling))
        self._ws[key] = ws
        return ws

    def _forward_split(self, x, w1, w2, w3):
        """``precision="bf16x3"``: the reference's fp32 arithmetic (srgan_train.py:525-576) at tensor-core speed for the
        convolutions that hold 91 % of the FLOPs. Stem (fp32 CUDA cores) -> trunk and both upsample convs in split-bf16
        (csrc/umma_trunk.cu, dbm_trunk_umma_split: hi + lo bf16 terms of every activation and filter, three MMAs per K
        chunk, fp32 accumulation and residual stream) -> deformable layers in fp32."""
        n, _, h, w = x.shape
        H, W = h - 2, w - 2
        if self.c_model_api and self.out_channels == 1:
            # the same sequence composed in C++ (csrc/gen_api.cu, dbm_gen_set_precision(gen, 1)): bit-identical
            return self._forward_c_api(x, w1, w2, w3)
        pk = self._pack(self.PACK_SPLIT)
        ws = self._split_workspace(n, H, W, pk)
        st = ops.stream()
        a0 = ops.empty(n, 128, H, W)
        self._stem_fp32(x, w1, w2, w3, a0)
        ops.call("dbm_nchw_to_slab8_split", a0.data_ptr(), 0, ws["s0"].data_ptr(), n, 128, H, W, st)
        del a0
        cat = ws["cat"]
        t, c, f = ws["tables"], ws["counts"], ws["flags"]
        ops.call("dbm_trunk_umma_split", t[0].data_ptr(), c[0], n, H, W, ws["s0"].data_ptr(), 16, cat[0].data_ptr(),
                 cat[1].data_ptr(), cat[0].shape[1] // 2, f[0].data_ptr(), st)
        u1, u2 = ws["u1"], ws["u2"]
        ops.call("dbm_trunk_umma_split", t[1].data_ptr(), 1, n, 2 * H, 2 * W, u1.data_ptr(), 8, u1.data_ptr(),
                 u1.data_ptr(), 8, f[1].data_ptr(), st)
        ops.call("dbm_trunk_umma_split", t[2].data_ptr(), 1, n, 4 * H, 4 * W, u2.data_ptr(), 8, u2.data_ptr(),
                 u2.data_ptr(), 8, f[2].data_ptr(), st)
        # deformable layers (srgan_train.py:572-574) in fp32, image by image (the fp32 sampler keeps a 576-row cols buffer)
        P = self.p
        y = ops.empty(n, self.out_channels, 4 * H, 4 * W)
        c2 = ops.empty(1, 64, 4 * H, 4 * W)
        per = 64 * 16 * H * W   # floats of one image in c2f (slab8f)
        for i in range(n):
            ops.call("dbm_slab8f_to_nchw", ws["c2f"].data_ptr() + 4 * per * i, c2.data_ptr(), 0, 1, 64, 4 * H, 4 * W, st)
            y[i:i + 1].copy_(self._deform_head_fp32(c2))
        return y

    def _deform_head_fp32(self, c2):
        """final_conv_layer1 (+ LeakyReLU) and final_conv_layer2 on c2 (n,64,4H,4W), fp32 CUDA cores."""
        P = self.p
        n = c2.shape[0]

        def conv(key, x_):
            wt = P[f"{key}/W"]
            out = ops.empty(n, wt.shape[0], x_.shape[2], x_.shape[3])
            ops.conv2d_fwd(x_, 0, 64, wt, P[f"{key}/b"], out, 0, 3, 1, 1, act=False)
            return out

        off1 = conv("final_conv_layer1/offset_conv", c2)
        d1, _ = ops.deform_conv_fwd(c2, off1, P["final_conv_layer1/deform_conv/W"], P["final_conv_layer1/deform_conv/b"],
                                    act=True, tc=False)
        del _
        off2 = conv("final_conv_layer2/offset_conv", d1)
        if self.out_channels == 1:
            y, _ = ops.deform1_conv_fwd(d1, off2, P["final_conv_layer2/deform_conv/W"], P["final_conv_layer2/deform_conv/b"])
        else:
            y, _ = ops.deform_conv_fwd(d1, off2, P["final_conv_layer2/deform_conv/W"], P["final_conv_layer2/deform_conv/b"],
                                       act=False)
        return y

    def _forward_bf16(self, x, w1, w2, w3):
        from . import flat
        P = self.p
        n, _, h, w = x.shape
        H, W = h - 2, w - 2
        bf = torch.bfloat16
        local = self.local_trunk and self.inter_channels == 32 and flat.local_trunk_fits(H, W)
        chain = self.local_trunk and self.inter_channels != 32 and flat.local_trunk_fits(H, W)
        if not local and not chain and self._c_forward_applies():
            return self._forward_c_api(x, w1, w2, w3)
        pk = self._pack(self.PACK_INFER_LOCAL if local else self.PACK_INFER)
        wt1, wts, bias128 = pk["stem"]
        if chain:
            # small tiles, wide dense blocks (inter_channels = 64, config 5): the flat layer chain on the padded-image
            # position axis instead of 32 x 16-pixel work units that a 9 x 9 tile fills to 16 %
            fc = self._ws.get(("chain", n, H, W))
            if fc is None:
                fc = self._ws[("chain", n, H, W)] = flat.FlatChainForward(self, n, H, W)
            fc.build(pk)
            ops.call("dbm_stem_fwd_flat", x.data_ptr(), w1.data_ptr(), w2.data_ptr(), w3.data_ptr(), wt1.data_ptr(),
                     wts.data_ptr(), bias128.data_ptr(), fc.s0.data_ptr(), n, h, w, ops.stream())
            a3 = fc.forward()
            u1 = ops.empty(n, 8, 2 * H, 2 * W, 8, dtype=bf)
            ops.nchw_to_slab8(ops.upsample2_fwd(a3), u1)
            ws = dict(u1=u1)
        elif local:
            # small tiles (the reference's 11x11 training / doctest windows): stem -> flat layout -> the whole trunk
            # with the activations of an image resident in shared memory / TMEM
            ws = self._local_workspace(n, H, W, pk)
            ops.call("dbm_stem_fwd_flat", x.data_ptr(), w1.data_ptr(), w2.data_ptr(), w3.data_ptr(), wt1.data_ptr(),
                     wts.data_ptr(), bias128.data_ptr(), ws["s0"].data_ptr(), n, h, w, ops.stream())
            ops.call("dbm_trunk_local_fwd", ws["table"].data_ptr(), ws["count"], n, H, W, ws["s0"].data_ptr(),
                     ws["x"][0].data_ptr(), ws["x"][1].data_ptr(), ops.stream())
        else:
            ws = self._trunk_workspace(n, H, W)
            if self.stem_w1_tensor_core:
                # conv_on_X / W2 / W3: small fp32 direct convs; conv_on_W1 (99 % of the stem's FLOPs): tcgen05
                s2d = ops.empty(n, 40, h, w, 8, dtype=bf)
                ops.call("dbm_stem_w1_s2d", w1.data_ptr(), s2d.data_ptr(), n, h, w, ops.stream())
                ops.call("dbm_stem_fwd_slab8", x.data_ptr(), None, w2.data_ptr(), w3.data_ptr(), None,
                         wts.data_ptr(), bias128.data_ptr(), ws["s0"].data_ptr(), 16, 0, n, h, w, ops.stream())
                ops.call("dbm_conv3x3_umma_valid", s2d.data_ptr(), 40, 320, pk["stem_w1_tc"].data_ptr(),
                         P["input_block/conv_on_W1/b"].data_ptr(), n, h, w, ws["s0"].data_ptr(), 16, 4, ops.stream())
                del s2d
            else:
                ops.call("dbm_stem_fwd_slab8", x.data_ptr(), w1.data_ptr(), w2.data_ptr(), w3.data_ptr(), wt1.data_ptr(),
                         wts.data_ptr(), bias128.data_ptr(), ws["s0"].data_ptr(), 16, 0, n, h, w, ops.stream())
            self._run_trunk(ws, n, H, W)
        u1 = ws["u1"]
        u2 = ops.empty(n, 8, 4 * H, 4 * W, 8, dtype=bf)
        wq, bq = pk["post_upsample_conv_layer_1"]
        ops.conv3x3_umma(u1, 64, wq, bq, 64, act=True, up2=True, out=u2)
        f1 = ops.empty(n, 8, 4 * H, 4 * W, 8, dtype=bf)
        wq, bq = pk["post_upsample_conv_layer_2"]
        ops.conv3x3_umma(u2, 64, wq, bq, 64, act=True, out=f1)
        del u2
        # deformable layers: offset conv (tcgen05) -> gather + tcgen05 contraction / output dot product
        off_s = ops.empty(n, 8, 4 * H, 4 * W, 4)
        wq, bq = pk["final_conv_layer1/offset_conv"]
        ops.conv3x3_umma(f1, 64, wq, bq, 32, out_f32=off_s)
        d1 = ops.empty(n, 8, 4 * H, 4 * W, 8, dtype=bf)
        wq, bq = pk["final_conv_layer1/deform_conv"]
        if self.out_channels != 1:
            raise ValueError("the tensor-core path implements out_channels == 1 (the reference's only use)")
        # the output layer's tap projection (64 -> 9 planes) is computed in this layer's epilogue
        proj = ops.deform_conv_umma(f1, off_s, wq, bq, d1, act=True,
                                    next_out1_w=P["final_conv_layer2/deform_conv/W"] if self.fuse_out_projection else None)
        del f1
        wq, bq = pk["final_conv_layer2/offset_conv"]
        ops.conv3x3_umma(d1, 64, wq, bq, 32, out_f32=off_s)
        if proj is not None:
            return ops.deform_out1_sample(proj, off_s, P["final_conv_layer2/deform_conv/b"])
        return ops.deform_conv_out1(d1, off_s, P["final_conv_layer2/deform_conv/W"],
                                    P["final_conv_layer2/deform_conv/b"])


# ================================================================================================
# Discriminator
# ================================================================================================
class DiscriminatorModel(_Link):
    """Drop-in for srgan_train.DiscriminatorModel (srgan_train.py:591-699): logits (N,1), no sigmoid.

    ``train`` replaces chainer.global_config.train (srgan_train.py:1125, 1228): True = batch
    statistics + running-stat update, False = running statistics.
    """

    BN_EPS = 1e-5
    BN_DECAY = 0.9

    def __init__(self, *, precision: str = "bf16", seed: int = 1, init_scale: float = 0.1):
        """``precision``: "bf16" = conv_layer1..9 (99 % of the FLOPs) on the tcgen05 tensor cores (bf16 operands,
        fp32 accumulation; flat.FlatConv, the 4x4 stride-2 layers as 3x3 GEMMs over space-to-depth phases);
        "fp32" = exact CUDA-core path. conv_layer0, BatchNormalization, LeakyReLU and the two Linear layers are
        fp32 in both."""
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        self.precision = precision
        self._tc_images, self._tc, self._tc_packed_version, self._tc_pack_table = None, {}, -1, None
        self._slot = 0
        shapes = layout.discriminator_shapes()
        super().__init__(shapes, layout.init_values(shapes, seed, init_scale))
        self.persistent = OrderedDict()
        for k, shp in layout.discriminator_persistents().items():
            self.persistent[k] = ops.zeros(*shp)
            if k.endswith("avg_var"):
                ops.fill(self.persistent[k], 1.0)
        self.bn_N = {i: 0 for i in range(1, 10)}
        self.train = True
        self._ctx = None

    def load_npz(self, file, strict: bool = True):
        npz_io.load_npz(file, self, strict=strict)
        return self

    def save_npz(self, file, compression: bool = True):
        npz_io.save_npz(file, self, compression=compression)

    def __call__(self, x, train: Optional[bool] = None):
        return self.forward(x, train=train)

    def forward(self, x, train: Optional[bool] = None, save: bool = False, groups: int = 1) -> Variable:
        """``groups`` > 1: the batch is ``groups`` independent passes stacked along N (the discriminator step feeds
        D(real) and D(fake), srgan_train.py:1145-1146): convolutions and linear layers run once over the whole
        stack, BatchNormalization takes its batch statistics (and updates the running ones, in order) per group --
        the same values as separate calls, half the kernel launches."""
        train = self.train if train is None else bool(train)
        x = as_device(x)
        if x.dim() != 4 or tuple(x.shape[1:]) != (1, 36, 36):
            # linear_1 is initialised for 512 inputs, i.e. 36x36 images (srgan_train.py:646, 693)
            raise ValueError(f"DiscriminatorModel expects (N,1,36,36) input, got {tuple(x.shape)}")
        P = self.p
        n = x.shape[0]
        if groups < 1 or n % groups:
            raise ValueError(f"batch of {n} does not split into {groups} groups")
        ng = n // groups
        acts = [x]
        pres = []
        a = ops.empty(n, 64, 36, 36)
        ops.conv2d_fwd(x, 0, 1, P["conv_layer0/W"], P["conv_layer0/b"], a, 0, 3, 1, 1, act=True)
        acts.append(a)
        stats = []
        hcur = 36
        cin = 64
        tc = self._tc_convs(n) if self.precision == "bf16" else None
        slot = 2   # forward inputs are kept per slot: 0 / 1 alternate for saved passes, 2 = no backward follows
        if save:
            slot = self._slot
            self._slot ^= 1
        for i in range(1, 10):
            cout, k, s = layout.DISC_CONVS[i]
            ho, _ = ops.conv_out_hw(hcur, hcur, k, s, 1)
            if tc is not None:
                z = tc[i].forward(acts[-1], slot)
            else:
                z = ops.empty(n, cout, ho, ho)
                ops.conv2d_fwd(acts[-1], 0, cin, P[f"conv_layer{i}/W"], None, z, 0, k, s, 1)
            y = ops.empty(n, cout, ho, ho)
            mean, invstd = ops.empty(groups, cout), ops.empty(groups, cout)
            # all groups in one pair of launches (statistics per group, running statistics updated in group order)
            ops.call("dbm_bn_lrelu_fwd_groups_f32", z.data_ptr(), y.data_ptr(), P[f"batch_norm{i}/gamma"].data_ptr(),
                     P[f"batch_norm{i}/beta"].data_ptr(), self.persistent[f"batch_norm{i}/avg_mean"].data_ptr(),
                     self.persistent[f"batch_norm{i}/avg_var"].data_ptr(), mean.data_ptr(), invstd.data_ptr(), groups, ng,
                     cout, ho * ho, self.BN_EPS, self.BN_DECAY, int(train), ops.stream())
            # batch_norm{i}/N: Chainer increments it in finetune mode only, which the reference never enters
            # (srgan_train.py:1125, 1228 toggle `train` alone) -> the loaded value (0 by default) is kept as is
            pres.append(z)
            stats.append((mean, invstd))
            acts.append(y)
            hcur, cin = ho, cout
        flat = acts[-1].view(n, 512)
        l1 = ops.empty(n, 100)
        ops.gemm(flat, 512, 1, 0, P["linear_1/W"], 1, 512, 0, l1, 100, 1, 0, P["linear_1/b"], n, 100, 512, act=True)
        out = ops.empty(n, 1)
        ops.gemm(l1, 100, 1, 0, P["linear_2/W"], 1, 100, 0, out, 1, 1, 0, P["linear_2/b"], n, 1, 100)
        if save:
            if not train:
                raise ValueError("backward through eval-mode BatchNormalization is not needed by the reference")
            self._ctx = dict(acts=acts, pres=pres, stats=stats, l1=l1, n=n, tc=tc, slot=slot, groups=groups)
        return Variable(out)

    def _tc_convs(self, n):
        from . import flat
        if self._tc_images is None:
            self._tc_images = {i: flat.ConvImages(self.p[f"conv_layer{i}/W"]) for i in range(1, 10)}
        if self._tc_packed_version != self.version:
            self._tc_pack_table = flat.pack_images(list(self._tc_images.values()), self._tc_pack_table)
            self._tc_packed_version = self.version
        tc = self._tc.get(n)
        if tc is None:
            tc, h = {}, 36
            for i in range(1, 10):
                _, k, s = layout.DISC_CONVS[i]
                tc[i] = flat.FlatConv(self._tc_images[i], self.g[f"conv_layer{i}/W"], n, h, h, nslots=3)
                h = ops.conv_out_hw(h, h, k, s, 1)[0]
            self._tc[n] = tc
        return tc

    def backward(self, dlogit: torch.Tensor, on_ready=None):
        """Accumulates parameter gradients for the most recent ``forward(save=True)`` given
        d(loss)/d(logits) (N,1); replaces d_loss.backward() (srgan_train.py:1163). ``on_ready(lo, hi)``:
        see GeneratorModel.backward (pass it only on the LAST backward of a step: the real and fake
        passes accumulate into the same buffer)."""
        if self._ctx is None:
            raise RuntimeError("backward() needs a preceding forward(save=True)")
        ready = (lambda *pre: on_ready(*self.grad_range(pre))) if on_ready is not None else (lambda *pre: None)
        c = self._ctx
        P, G = self.p, self.g
        n = c["n"]
        acts, pres, stats, l1 = c["acts"], c["pres"], c["stats"], c["l1"]
        dlogit = dlogit.contiguous()
        # linear_2
        ops.gemm(dlogit, 1, 1, 0, l1, 100, 1, 0, G["linear_2/W"], 100, 1, 0, None, 1, 100, n, accumulate=1)
        ops.call("dbm_bias_grad_f32", dlogit.data_ptr(), 1, G["linear_2/b"].data_ptr(), n, 1, 1, ops.stream())
        dl1 = ops.empty(n, 100)
        ops.gemm(dlogit, 1, 1, 0, P["linear_2/W"], 100, 1, 0, dl1, 100, 1, 0, None, n, 100, 1)
        ops.lrelu_bwd(dl1, 0, l1, 0, dl1, 0, 100)
        # linear_1: dW[o, i] += sum_n dl1[n, o] * flat[n, i]
        flat = acts[-1].view(n, 512)
        ops.gemm(dl1, 1, 100, 0, flat, 512, 1, 0, G["linear_1/W"], 512, 1, 0, None, 100, 512, n, accumulate=1)
        ops.call("dbm_bias_grad_f32", dl1.data_ptr(), 100, G["linear_1/b"].data_ptr(), n, 100, 1, ops.stream())
        dflat = ops.empty(n, 512, 1, 1)
        ops.gemm(dl1, 100, 1, 0, P["linear_1/W"], 512, 1, 0, dflat, 512, 1, 0, None, n, 512, 100)
        dy = dflat
        # The nine tensor-core weight gradients (+ their reductions) feed only the optimizer: they run on a side stream
        # beside the BatchNorm / data-gradient chain -- ~100 us per layer off this model's critical path -- and are
        # joined before each gradient bucket is handed on.
        cur = torch.cuda.current_stream()
        wg = ops._aux_stream2() if c.get("tc") is not None else None
        for i in range(9, 0, -1):
            cout, k, s = layout.DISC_CONVS[i]
            z, y = pres[i - 1], acts[i + 1]
            mean, invstd = stats[i - 1]
            hw = z.shape[2] * z.shape[3]
            dz = ops.empty(*z.shape)
            groups = c.get("groups", 1)
            ng = n // groups
            scratch = ops.empty(groups, 2 * cout)
            ops.call("dbm_bn_lrelu_bwd_groups_f32", z.data_ptr(), y.data_ptr(), dy.data_ptr(), dz.data_ptr(),
                     P[f"batch_norm{i}/gamma"].data_ptr(), mean.data_ptr(), invstd.data_ptr(),
                     G[f"batch_norm{i}/gamma"].data_ptr(), G[f"batch_norm{i}/beta"].data_ptr(), scratch.data_ptr(),
                     groups, ng, cout, hw, ops.stream())
            xin = acts[i]
            cin = xin.shape[1]
            if c.get("tc") is not None:
                dx = c["tc"][i].backward(dz, c["slot"], wgrad_stream=wg)
            else:
                ops.conv2d_bwd_weight(xin, 0, cin, dz, 0, G[f"conv_layer{i}/W"], k, s, 1)
                dx = ops.empty(*xin.shape)
                ops.conv2d_bwd_data(dz, 0, P[f"conv_layer{i}/W"], dx, 0, cin, k, s, 1)
            dy = dx
            if i in (9, 5) and on_ready is not None:
                # Hand the finished buckets over ON the weight-gradient stream (after it has caught up with the
                # BatchNorm / linear gradients produced on this one): the data-gradient chain -- the critical path of
                # the whole training step -- never waits for a weight gradient. (Round 2: joining the streams here
                # stalled the chain for 0.7 ms behind the 512-channel layers' weight gradients.)
                with torch.cuda.stream(wg if wg is not None else cur):
                    if wg is not None:
                        wg.wait_stream(cur)
                    if i == 9:
                        ready("linear_", "conv_layer9/", "batch_norm9/")
                    else:
                        ready("conv_layer5/", "batch_norm5/", "conv_layer6/", "batch_norm6/", "conv_layer7/",
                              "batch_norm7/", "conv_layer8/", "batch_norm8/")
        # conv_layer0 + LeakyReLU
        ops.lrelu_bwd(dy, 0, acts[1], 0, dy, 0, 64)
        ops.conv2d_bwd_weight(acts[0], 0, 1, dy, 0, G["conv_layer0/W"], 3, 1, 1, db=G["conv_layer0/b"])
        if wg is not None:
            cur.wait_stream(wg)
        ready("conv_layer0/", "conv_layer1/", "batch_norm1/", "conv_layer2/", "batch_norm2/", "conv_layer3/",
              "batch_norm3/", "conv_layer4/", "batch_norm4/")
        self._ctx = None
