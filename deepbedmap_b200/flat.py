"""Host side of the tensor-core TRAINING trunk (csrc/umma_flat.cu): buffers in the flat-padded slab
layout and the launch / unit tables of the forward chain, the data-gradient chain and the batched
weight-gradient of the generator trunk (pre-residual conv, 3*nb residual dense blocks, post-residual
conv: srgan_train.py:292-358, 393-404, 467-486, 541-551, and their autograd in g_loss.backward(), :1256).

Arithmetic: bf16 operands (activations, gradients wrt activations, filters), fp32 TMEM accumulation,
fp32 residual stream and fp32 accumulation of the dense-block gradients; fp32 master weights/gradients.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import ops

# mirrors of the structs in csrc/umma_flat.cu
EPI_DTYPE = np.dtype([("bias", "<u8"), ("add1", "<u8"), ("add2", "<u8"), ("mask", "<u8"), ("out_f32", "<u8"),
                      ("out_bf16", "<u8"), ("s1", "<f4"), ("beta", "<f4"), ("beta2", "<f4"), ("out_scale", "<f4"),
                      ("act", "<i4"), ("pad", "<i4")])
assert EPI_DTYPE.itemsize == 72
LAUNCH_DTYPE = np.dtype([("in", "<u8"), ("wpacked", "<u8"), ("cin", "<i4"), ("nout", "<i4"), ("ny", "<i4"), ("pad", "<i4"),
                         ("w_chunk_stride", "<i8"), ("blk", EPI_DTYPE, (6,))])
assert LAUNCH_DTYPE.itemsize == 472
WGRAD_UNIT_DTYPE = np.dtype([("act", "<u8"), ("gout", "<u8"), ("partial", "<u8"), ("blk0", "<i4"), ("nblk", "<i4"),
                             ("nslab", "<i4"), ("tapmask", "<i4"), ("pad", "<i4", (2,))])
assert WGRAD_UNIT_DTYPE.itemsize == 48
WGRAD_REDUCE_DTYPE = np.dtype([("partial", "<u8"), ("dw", "<u8"), ("split_stride", "<i8"), ("nsplit", "<i4"),
                               ("cin_total", "<i4"), ("c0", "<i4"), ("o0", "<i4"), ("nch", "<i4"), ("mode", "<i4")])
assert WGRAD_REDUCE_DTYPE.itemsize == 48
BIAS_GRAD_DTYPE = np.dtype([("gout", "<u8"), ("db", "<u8")])
# csrc/umma_local.cu LocalPass
LOCAL_PASS_DTYPE = np.dtype([("w", "<u8"), ("bias", "<u8"), ("save", "<u8"), ("out_f32", "<u8"), ("mask", "<u8"),
                             ("add_f32", "<u8"), ("slab0", "<i4"), ("nk", "<i4"), ("N", "<i4"), ("col0", "<i4"),
                             ("type", "<i4"), ("ecol", "<i4"), ("out_slab", "<i4"), ("rr", "<i4"), ("beta", "<f4"),
                             ("scale", "<f4"), ("first", "<i4"), ("pad", "<i4")])
assert LOCAL_PASS_DTYPE.itemsize == 96
LOC_PRE, LOC_ACT, LOC_RDB, LOC_POST, LOC_BPOST, LOC_BMASK, LOC_BD1, LOC_BPRE = range(8)


def local_trunk_fits(H: int, W: int) -> bool:
    """An image with its zero border is one M=128 UMMA tile: the image-resident kernel applies."""
    return (H + 2) * (W + 2) <= 128


def local_pass(**kw):
    e = np.zeros((), dtype=LOCAL_PASS_DTYPE)
    e["scale"] = 1.0
    for k, v in kw.items():
        e[k] = v
    return e


def local_forward_table(model, pk, nrdb, beta, cat_ptr=None, out_f32=0, up2_out=0):
    """Pass table of dbm_trunk_local_fwd for ``model``'s packed operands. ``cat_ptr(j, c)``: flat bf16 address of
    channel c of dense-block buffer j (None: inference, nothing is kept); ``out_f32``: flat fp32 slab4 output;
    ``up2_out``: bf16 slab8 (n, 8, 2H, 2W, 8) output, nearest-upsampled x2 (inference head)."""
    P = model.p
    save = (lambda j, c: cat_ptr(j, c)) if cat_ptr is not None else (lambda j, c: 0)
    passes = [local_pass(w=pk["pre_residual_conv_layer@trunk"][0].data_ptr(),
                         bias=P["pre_residual_conv_layer/b"].data_ptr(), save=save(0, 0), slab0=0, nk=8, N=64, col0=0,
                         type=LOC_PRE, ecol=0, out_slab=0, first=1)]
    for j in range(nrdb):
        r = j % 3 + 1
        pre = model._rdb_prefix(j // 3, r)
        for s in range(5):
            last = s == 4
            passes.append(local_pass(
                w=pk[f"{pre}/stat{s}"].data_ptr(), bias=P[f"{pre}/conv_layer{s + 1}/b"].data_ptr(),
                save=save(j + 1, 0) if last else save(j, 64 + 32 * s), slab0=0 if s == 0 else 8 + 4 * (s - 1),
                nk=4 if s == 0 else 2, N=192 - 32 * s, col0=32 * s, type=LOC_RDB if last else LOC_ACT, ecol=32 * s,
                out_slab=0 if last else 8 + 4 * s, rr=int(last and r == 3), beta=beta, first=int(s == 0)))
    passes.append(local_pass(w=pk["post_residual_conv_layer@trunk"][0].data_ptr(),
                             bias=P["post_residual_conv_layer/b"].data_ptr(), out_f32=out_f32, save=up2_out, slab0=0,
                             nk=4, N=64,
                             col0=0, type=LOC_POST, ecol=0, first=1))
    return np.ascontiguousarray(np.stack(passes))
PARTIAL_FLOATS = 9 * 32 * 128


def geometry(n: int, h: int, w: int) -> dict:
    """{P, tiles, G0, Pg, R} of the flat-padded layout for n images of h x w pixels (from the library,
    so host tables and kernels cannot disagree)."""
    out = (ctypes.c_int * 5)()
    ops.call("dbm_flat_geometry", n, h, w, ctypes.cast(out, ctypes.c_void_p))
    return dict(P=out[0], tiles=out[1], G0=out[2], Pg=out[3], R=out[4])


def geometry_host(n: int, h: int, w: int) -> dict:
    """The same formula in Python (checked against the library by tests/test_cabi.py)."""
    wp = w + 2
    P = n * (h + 2) * wp
    tiles = (P + 127) // 128
    halo = wp + 1
    g0 = (halo + 7) & ~7
    return dict(P=P, tiles=tiles, G0=g0, Pg=g0 + tiles * 128 + g0, R=128 + 2 * halo)


def split_blocks(tiles: int, nsplit: int):
    """[(blk0, nblk)] covering range(tiles) in nsplit near-equal contiguous ranges (empty ranges dropped)."""
    nsplit = max(1, min(nsplit, tiles))
    base, rem = divmod(tiles, nsplit)
    out, b = [], 0
    for s in range(nsplit):
        k = base + (1 if s < rem else 0)
        out.append((b, k))
        b += k
    return out


def s2d_tap_mask(c0: int, nch: int, C: int) -> int:
    """Taps (bit t = tap t = ky * 3 + kx of the embedding 3x3 filter) that are not structurally zero for the phase
    channels [c0, c0 + nch) of a 4x4 stride-2 filter over C input channels (phase = channel // C = py * 2 + px):
    filter row 2 (ky - 1) + py + 1 must lie in 0..3, i.e. ky in {1, 2} for py = 0 and {0, 1} for py = 1; same in x."""
    mask = 0
    for ph in range(c0 // C, (c0 + nch - 1) // C + 1):
        py, px = ph >> 1, ph & 1
        for ky in ((1, 2) if py == 0 else (0, 1)):
            for kx in ((1, 2) if px == 0 else (0, 1)):
                mask |= 1 << (ky * 3 + kx)
    return mask


def chunk_channels(cin: int, chunk: int = 128):
    """[(c0, nch)] input-channel chunks of a weight-gradient GEMM (M = 128 channels per UMMA tile)."""
    return [(c0, min(chunk, cin - c0)) for c0 in range(0, cin, chunk)]


def rdb_plan(nrdb: int, beta: float):
    """Per residual dense block j (0-based, r = j % 3 + 1 within its RRDB): sigma_j = d(rdb_out)/d(x_{j+1})
    scale (beta for the third block of an RRDB, whose output is scaled again by the RRDB: :402), and the scale
    of the bf16 conv5 output gradient g5_j = beta * sigma_j * dX_{j+1} (:358)."""
    plan = []
    for j in range(nrdb):
        r = j % 3 + 1
        sigma = beta if r == 3 else 1.0
        plan.append(dict(j=j, r=r, sigma=sigma, g5_scale=beta * sigma))
    return plan


def epi(**kw):
    """One FlatEpiBlock record; scales default to 1."""
    e = np.zeros((), dtype=EPI_DTYPE)
    e["s1"] = 1.0
    e["beta"] = 1.0
    e["beta2"] = 1.0
    e["out_scale"] = 1.0
    for k, v in kw.items():
        e[k] = v
    return e


def launch(inp_ptr, wq, cin, nout, blocks):
    """One FlatLaunch record: a 3x3 conv of ``cin`` channels at ``inp_ptr`` with packed filter ``wq``, N = ``nout``,
    one epilogue block per 32 output channels."""
    L = np.zeros((), dtype=LAUNCH_DTYPE)
    L["in"] = inp_ptr
    L["wpacked"] = wq.data_ptr()
    L["cin"] = cin
    L["nout"] = nout
    L["ny"] = 1
    assert len(blocks) == nout // 32
    for b, e in enumerate(blocks):
        L["blk"][b] = e
    return L


def forward_chain(model, pk, Pg, s0, cat, x, a3f):
    """Launch records of the trunk's forward (srgan_train.py:541-551) on the flat-padded layout, ``Pg`` positions per
    channel: the pre-residual conv from the stem output ``s0``, the 3 * nb residual dense blocks, the post-residual conv
    with the skip a1 into ``a3f``. Dense block j reads [a0 | a1..a4] from ``cat(j)`` (filling a1..a4 there) and writes
    its bf16 output into ``cat(j + 1)``; ``x(j)`` is the fp32 residual stream into block j (``x(0)`` = a1)."""
    beta, g = model.residual_scaling, model.inter_channels
    pb = lambda t, c=0: t.data_ptr() + 2 * c * Pg
    pf = lambda t, c=0: t.data_ptr() + 4 * c * Pg
    nrdb = 3 * model.num_residual_blocks
    wq, bq = pk["pre_residual_conv_layer@trunk"]
    tab = [launch(pb(s0), wq, 128, 64, [
        epi(bias=bq.data_ptr() + 128 * b, act=1, out_f32=pf(x(0), 32 * b), out_bf16=pb(cat(0), 32 * b)) for b in range(2)])]
    for j in range(nrdb):
        r = j % 3 + 1
        pre = model._rdb_prefix(j // 3, r)
        for k in (1, 2, 3, 4):
            cin = 64 + g * (k - 1)
            wq, bq = pk[f"{pre}/conv_layer{k}@trunk"]
            tab.append(launch(pb(cat(j)), wq, cin, g, [
                epi(bias=bq.data_ptr() + 128 * b, act=1, out_bf16=pb(cat(j), cin + 32 * b)) for b in range(g // 32)]))
        wq, bq = pk[f"{pre}/conv_layer5@trunk"]
        blocks = []
        for b in range(2):
            kw = dict(bias=bq.data_ptr() + 128 * b, add1=pf(x(j), 32 * b), s1=1.0, beta=beta,
                      out_f32=pf(x(j + 1), 32 * b), out_bf16=pb(cat(j + 1), 32 * b))
            if r == 3:   # out = rrdb_in + beta * (x + beta * a5)  (srgan_train.py:358, 402)
                kw.update(add2=pf(x(j - 2), 32 * b), beta2=beta)
            blocks.append(epi(**kw))
        tab.append(launch(pb(cat(j)), wq, 64 + 4 * g, 64, blocks))
    wq, bq = pk["post_residual_conv_layer@trunk"]
    tab.append(launch(pb(cat(nrdb)), wq, 64, 64, [
        epi(bias=bq.data_ptr() + 128 * b, add1=pf(x(0), 32 * b), s1=1.0, beta=1.0, out_f32=pf(a3f, 32 * b))
        for b in range(2)]))
    return tab


class FlatTrunk:
    """Buffers + tables of the tensor-core training trunk for one (batch, H, W)."""

    NSPLIT = 3

    def __init__(self, model, n: int, H: int, W: int):
        if model.inter_channels not in (32, 64):
            raise ValueError("the tensor-core training trunk implements inter_channels 32 or 64")
        self.model = model
        self.G = G = model.inter_channels   # dense-block growth (srgan_train.py:283-284)
        self.cc = cc = 64 + 4 * G           # channels of a dense-block buffer [a0 (64) | a1 .. a4 (G each)]
        self.n, self.H, self.W = n, H, W
        self.geom = geometry(n, H, W)
        Pg = self.geom["Pg"]
        self.Pg = Pg
        nrdb = 3 * model.num_residual_blocks
        self.nrdb = nrdb
        bf = torch.bfloat16
        zb = lambda c: torch.zeros(c // 8, Pg, 8, dtype=bf, device="cuda")
        zf = lambda c: torch.zeros(c // 4, Pg, 4, dtype=torch.float32, device="cuda")
        self.s0 = zb(128)
        self.cat = [zb(cc) for _ in range(nrdb + 1)]        # cat[j][:64] = bf16 input of RDB j, slots a1..a4 follow
        self.gcat = [zb(cc) for _ in range(nrdb)]           # [g1 | g2 | g3 | g4 (G each) | g5 (64)] gradients wrt conv outputs
        self.x0 = zf(64)
        self.xring = [zf(64) for _ in range(4)]
        self.a3f = zf(64)
        self.gpost, self.gpre = zb(64), zb(64)
        self.da3f = zf(64)
        self.dX = [zf(64) for _ in range(4)]
        self.dcat = zf(cc)
        self.da0f = zf(128)
        self._pack_gen = -1
        self._built_beta = None

    # ---- pointer helpers (block = 32 channels starting at channel c) ----
    def _pb(self, t, c=0):
        return t.data_ptr() + 2 * c * self.Pg

    def _pf(self, t, c=0):
        return t.data_ptr() + 4 * c * self.Pg

    def _x(self, j):
        return self.x0 if j == 0 else self.xring[j % 4]

    def _launches(self, inp_ptr, slices, cin, blocks):
        """One conv whose N exceeds the kernels' 192 columns as consecutive launches over N-slices of its operand
        (``slices``: [(n0, width, packed image)], model._pack's ``@dgrad_slices``); ``blocks`` cover all of N."""
        out = []
        for n0, width, img in slices:
            out.append(launch(inp_ptr, img, cin, width, blocks[n0 // 32:(n0 + width) // 32]))
        return out

    def build(self, pk):
        """(Re)build every table against the model's packed-operand buffers ``pk`` (model._pack())."""
        m = self.model
        beta = m.residual_scaling
        if self._pack_gen == m._pack_gen and self._built_beta == beta:
            return
        P, Gr = m.p, m.g
        G, cc = self.G, self.cc
        nrdb = self.nrdb
        pb, pf = self._pb, self._pf
        plan = rdb_plan(nrdb, beta)
        bwd = []
        convs = []  # (key, act tensor, cin, g tensor, g channel0, cout) for the weight / bias gradients

        fwd = forward_chain(m, pk, self.Pg, self.s0, lambda j: self.cat[j], self._x, self.a3f)

        # ---------------- data-gradient chain ----------------
        dX = lambda j: self.dX[j % 4]
        gb = G // 32                       # 32-channel epilogue blocks per dense-block slot
        nb5 = cc // 32                     # blocks of conv5's data gradient d[a0 .. a4]
        wq = pk["post_residual_conv_layer@dgrad"]
        bwd.append(launch(pb(self.gpost), wq, 64, 64, [
            epi(out_f32=pf(dX(nrdb), 32 * b), out_bf16=pb(self.gcat[nrdb - 1], 4 * G + 32 * b),
                out_scale=plan[nrdb - 1]["g5_scale"]) for b in range(2)]))
        convs.append(("post_residual_conv_layer", self.cat[nrdb], 64, self.gpost, 0, 64))
        for d in reversed(plan):
            j, r, sigma = d["j"], d["r"], d["sigma"]
            pre = m._rdb_prefix(j // 3, r)
            cat, gcat = self.cat[j], self.gcat[j]
            # conv5: g5 (64) -> d[a0..a4] (64 + 4G); + skip sigma * dX_{j+1} on a0; slot a4 finalised -> g4
            blocks = []
            for b in range(nb5):
                kw = {}
                if b < 2:
                    kw.update(add1=pf(dX(j + 1), 32 * b), s1=sigma, beta=1.0)
                    if j == 0:  # the skip a3 = a1 + post_res(...) (:551) reaches a1 = input of RDB 0
                        kw.update(add2=pf(self.da3f, 32 * b), beta2=1.0)
                if b < nb5 - gb:
                    kw.update(out_f32=pf(self.dcat, 32 * b))
                else:
                    kw.update(mask=pb(cat, 32 * b), out_bf16=pb(gcat, 3 * G + 32 * (b - (nb5 - gb))))
                blocks.append(epi(**kw))
            bwd.extend(self._launches(pb(gcat, 4 * G), pk[f"{pre}/conv_layer5@dgrad_slices"], 64, blocks))
            convs.append((f"{pre}/conv_layer5", cat, cc, gcat, 4 * G, 64))
            for k in (4, 3, 2):
                nout = 64 + G * (k - 1)
                nbk = nout // 32
                blocks = []
                for b in range(nbk):
                    kw = dict(add1=pf(self.dcat, 32 * b), s1=1.0, beta=1.0)
                    if b < nbk - gb:
                        kw.update(out_f32=pf(self.dcat, 32 * b))
                    else:  # slot a_{k-1} is final: apply lrelu' and emit the bf16 operand of the next dgrad
                        kw.update(mask=pb(cat, 32 * b), out_bf16=pb(gcat, G * (k - 2) + 32 * (b - (nbk - gb))))
                    blocks.append(epi(**kw))
                bwd.extend(self._launches(pb(gcat, G * (k - 1)), pk[f"{pre}/conv_layer{k}@dgrad_slices"], G, blocks))
                convs.append((f"{pre}/conv_layer{k}", cat, nout, gcat, G * (k - 1), G))
            blocks = []
            for b in range(2):
                kw = dict(add1=pf(self.dcat, 32 * b), s1=1.0, beta=1.0)
                if r == 1:  # RRDB skip: d x_{3i} += d x_{3i+3} (:402)
                    kw.update(add2=pf(dX(j + 3), 32 * b), beta2=1.0)
                if j > 0:
                    kw.update(out_f32=pf(dX(j), 32 * b), out_bf16=pb(self.gcat[j - 1], 4 * G + 32 * b),
                              out_scale=plan[j - 1]["g5_scale"])
                else:   # a1 = lrelu(pre_res(a0)) (:541-544)
                    kw.update(mask=pb(self.cat[0], 32 * b), out_bf16=pb(self.gpre, 32 * b))
                blocks.append(epi(**kw))
            bwd.append(launch(pb(gcat, 0), pk[f"{pre}/conv_layer1@dgrad"], G, 64, blocks))
            convs.append((f"{pre}/conv_layer1", cat, 64, gcat, 0, G))
        bwd.append(launch(pb(self.gpre), pk["pre_residual_conv_layer@dgrad"], 64, 128,
                          [epi(out_f32=pf(self.da0f, 32 * b)) for b in range(4)]))
        convs.append(("pre_residual_conv_layer", self.s0, 128, self.gpre, 0, 64))

        # ---------------- weight / bias gradient tables ----------------
        splits = split_blocks(self.geom["tiles"], self.NSPLIT)
        units, reduces, biases = [], [], []
        for key, act, cin, gt, g0, cout in convs:
            for half in range(cout // 32):
                biases.append((pb(gt, g0 + 32 * half), Gr[f"{key}/b"].data_ptr() + 128 * half))
                for c0, nch in chunk_channels(cin):
                    first = len(units)
                    for blk0, nblk in splits:
                        units.append((pb(act, c0), pb(gt, g0 + 32 * half), len(units), blk0, nblk, nch // 8, 0, (0, 0)))
                    reduces.append((first, Gr[f"{key}/W"].data_ptr(), PARTIAL_FLOATS, len(splits), cin, c0, 32 * half,
                                    nch, 0))
        need = len(units) * PARTIAL_FLOATS
        if getattr(self, "partial", None) is None or self.partial.numel() < need:
            self.partial = torch.empty(need, dtype=torch.float32, device="cuda")
        base = self.partial.data_ptr()
        u = np.array(units, dtype=WGRAD_UNIT_DTYPE)
        u["partial"] = base + u["partial"] * np.uint64(PARTIAL_FLOATS * 4)
        rd = np.array(reduces, dtype=WGRAD_REDUCE_DTYPE)
        rd["partial"] = base + rd["partial"] * np.uint64(PARTIAL_FLOATS * 4)
        bg = np.array(biases, dtype=BIAS_GRAD_DTYPE)
        dev = lambda a: torch.from_numpy(a.view(np.uint8).reshape(-1).copy()).cuda()
        self.units_dev, self.n_units = dev(u), len(u)
        self.reduce_dev, self.n_reduce = dev(rd), len(rd)
        self.bias_dev, self.n_bias = dev(bg), len(bg)
        self.fwd = np.ascontiguousarray(np.stack(fwd))
        self.bwd = np.ascontiguousarray(np.stack(bwd))
        # device copies + dependency flags of the persistent chain launches (dbm_flat_conv3x3_chain)
        self.fwd_dev, self.bwd_dev = dev(self.fwd), dev(self.bwd)
        self.flags = torch.zeros(max(len(fwd), len(bwd)) * self.geom["tiles"], dtype=torch.int32, device="cuda")
        self.flops_fwd = float(sum(2.0 * 9 * int(L["cin"]) * int(L["nout"]) for L in fwd)) * self.n * self.H * self.W
        # image-resident forward (csrc/umma_local.cu) when a padded image is one UMMA tile
        self.local_dev = None
        if G == 32 and local_trunk_fits(self.H, self.W):
            tab = local_forward_table(m, pk, nrdb, beta, cat_ptr=lambda j, c: pb(self.cat[j], c), out_f32=pf(self.a3f))
            self.local_dev, self.n_local = dev(tab), len(tab)
            if getattr(self, "x_scratch", None) is None:
                self.x_scratch = torch.empty(2, self.n * 16 * 128 * 4, dtype=torch.float32, device="cuda")
            # data-gradient chain, image-resident: same passes as ``bwd`` above (conv5's gradient opens the block's
            # accumulator d[a0..a4], conv4..conv1's add onto its leading columns); operand slabs in shared memory:
            # g5 -> 0..7, g4 -> 8, g3 -> 12, g2 -> 16, g1 -> 20
            gp = lambda key: pk[key].data_ptr()
            bt = [local_pass(w=gp("post_residual_conv_layer@dgrad"), save=pb(self.gcat[nrdb - 1], 128), slab0=0, nk=4,
                             N=64, col0=0, type=LOC_BPOST, ecol=0, out_slab=0, scale=plan[nrdb - 1]["g5_scale"], first=1)]
            for d in reversed(plan):
                j, r, sigma = d["j"], d["r"], d["sigma"]
                pre = m._rdb_prefix(j // 3, r)
                cat, gcat = self.cat[j], self.gcat[j]
                bt.append(local_pass(w=gp(f"{pre}/conv_layer5@dgrad"), mask=pb(cat, 160), save=pb(gcat, 96), slab0=0, nk=4,
                                     N=192, col0=0, type=LOC_BMASK, ecol=160, out_slab=8, first=1))
                for k in (4, 3, 2):
                    nout = 64 + 32 * (k - 1)
                    bt.append(local_pass(w=gp(f"{pre}/conv_layer{k}@dgrad"), mask=pb(cat, nout - 32),
                                         save=pb(gcat, 32 * (k - 2)), slab0=8 + 4 * (4 - k), nk=2, N=nout, col0=0,
                                         type=LOC_BMASK, ecol=nout - 32, out_slab=8 + 4 * (5 - k), first=0))
                kw = dict(w=gp(f"{pre}/conv_layer1@dgrad"), slab0=20, nk=2, N=64, col0=0, type=LOC_BD1, ecol=0, out_slab=0,
                          beta=sigma, rr=int(r == 1), first=0)
                if j > 0:
                    kw.update(save=pb(self.gcat[j - 1], 128), scale=plan[j - 1]["g5_scale"])
                else:
                    kw.update(mask=pb(self.cat[0], 0), save=pb(self.gpre), add_f32=pf(self.da3f))
                bt.append(local_pass(**kw))
            bt.append(local_pass(w=gp("pre_residual_conv_layer@dgrad"), out_f32=pf(self.da0f), slab0=0, nk=4, N=128, col0=0,
                                 type=LOC_BPRE, ecol=0, first=1))
            self.local_bwd_dev, self.n_local_bwd = dev(np.ascontiguousarray(np.stack(bt))), len(bt)
        self._pack_gen = m._pack_gen
        self._built_beta = beta

    # ---- execution ----
    persistent = True   # one persistent launch per chain (False: one launch per layer, the A/B reference)
    local = True        # forward: image-resident kernel when the tile fits (False: the flat chain, the A/B reference)

    def _chain(self, table, table_dev):
        n, H, W = self.n, self.H, self.W
        if self.persistent:
            ops.call("dbm_flat_conv3x3_chain", table.ctypes.data, table_dev.data_ptr(), len(table), n, H, W, 0, 0,
                     self.flags.data_ptr(), ops.stream())
        else:
            ops.call("dbm_flat_conv3x3_seq", table.ctypes.data, len(table), n, H, W, 0, 0, ops.stream())

    def forward(self, a0_nchw: torch.Tensor) -> torch.Tensor:
        """a0 = stem output (n,128,H,W) fp32 -> a3 = a1 + post_res(trunk(a1)) (n,64,H,W) fp32 (:541-551);
        keeps the bf16 activations of every dense block for backward()."""
        n, H, W = self.n, self.H, self.W
        st = ops.stream()
        ops.call("dbm_flat_from_nchw", a0_nchw.data_ptr(), 128, self.s0.data_ptr(), None, 1.0, n, H, W, st)
        if self.local and self.local_dev is not None:
            ops.call("dbm_trunk_local_fwd", self.local_dev.data_ptr(), self.n_local, n, H, W, self.s0.data_ptr(),
                     self.x_scratch[0].data_ptr(), self.x_scratch[1].data_ptr(), st)
        else:
            self.model._pack(self.model.PACK_TRAIN_CHAIN)   # the chain reads the per-layer 16-channel images
            self._chain(self.fwd, self.fwd_dev)
        a3 = ops.empty(n, 64, H, W)
        ops.call("dbm_flat_to_nchw", self.a3f.data_ptr(), None, a3.data_ptr(), 64, n, H, W, st)
        return a3

    def backward(self, da3_nchw: torch.Tensor, wgrad_stream=None) -> torch.Tensor:
        """da3 (n,64,H,W) -> accumulates the trunk's weight/bias gradients into the model's flat_grad and
        returns d(loss)/d(a0) (n,128,H,W). ``wgrad_stream``: torch stream for the weight / bias gradient launches
        (they start after the data-gradient chain; the CALLER joins that stream before using the gradients)."""
        n, H, W = self.n, self.H, self.W
        st = ops.stream()
        ops.call("dbm_flat_from_nchw", da3_nchw.data_ptr(), 64, self.gpost.data_ptr(), self.da3f.data_ptr(), 1.0, n, H, W,
                 st)
        if self.local and self.local_dev is not None:
            ops.call("dbm_trunk_local_bwd", self.local_bwd_dev.data_ptr(), self.n_local_bwd, n, H, W,
                     self.gpost.data_ptr(), self.x_scratch[1].data_ptr(), st)
        else:
            self.model._pack(self.model.PACK_TRAIN_CHAIN)
            self._chain(self.bwd, self.bwd_dev)
        if wgrad_stream is not None:
            wgrad_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(wgrad_stream if wgrad_stream is not None else torch.cuda.current_stream()):
            ws = ops.stream()
            ops.call("dbm_flat_wgrad_ctas", self.units_dev.data_ptr(), self.n_units, n, H, W,
                     int(getattr(self.model, "trunk_wgrad_ctas", 0)), ws)
            ops.call("dbm_flat_wgrad_reduce", self.reduce_dev.data_ptr(), self.n_reduce, ws)
            ops.call("dbm_flat_bias_grad", self.bias_dev.data_ptr(), self.n_bias, n, H, W, ws)
        da0 = ops.empty(n, 128, H, W)
        ops.call("dbm_flat_to_nchw", self.da0f.data_ptr(), None, da0.data_ptr(), 128, n, H, W, st)
        return da0


class FlatChainForward:
    """Inference forward of the trunk (srgan_train.py:541-551) on the flat-padded layout through the persistent layer
    chain (dbm_flat_conv3x3_chain), for either dense-block width (inter_channels 32 or 64, srgan_train.py:283-284):
    the path of SMALL tiles -- an image with its border is at most one 128-position MMA tile -- when the image-resident
    kernel (inter_channels = 32 only) does not apply. On such tiles the tiled trunk kernel would use 81 of the 512 pixels
    of its 32 x 16 work units; here all padded images are one flat position axis."""

    def __init__(self, model, n: int, H: int, W: int):
        self.model, self.n, self.H, self.W = model, n, H, W
        self.geom = geometry(n, H, W)
        self.Pg = Pg = self.geom["Pg"]
        g = model.inter_channels
        self.cc = 64 + 4 * g
        bf = torch.bfloat16
        zb = lambda c: torch.zeros(c // 8, Pg, 8, dtype=bf, device="cuda")
        zf = lambda c: torch.zeros(c // 4, Pg, 4, dtype=torch.float32, device="cuda")
        self.s0 = zb(128)
        self.cat = [zb(self.cc), zb(self.cc)]
        self.x0 = zf(64)
        self.xring = [zf(64) for _ in range(4)]
        self.a3f = zf(64)
        self._key = None

    def _x(self, j):
        return self.x0 if j == 0 else self.xring[j % 4]

    def build(self, pk):
        m = self.model
        key = (m._pack_gen, m.residual_scaling)
        if self._key == key:
            return
        tab = forward_chain(m, pk, self.Pg, self.s0, lambda j: self.cat[j % 2], self._x, self.a3f)
        self.table = np.ascontiguousarray(np.stack(tab))
        self.table_dev = torch.from_numpy(self.table.view(np.uint8).reshape(-1).copy()).cuda()
        self.flags = ops.empty(len(tab) * self.geom["tiles"], dtype=torch.int32)
        self._key = key

    def forward(self) -> torch.Tensor:
        """s0 (flat bf16 stem output, filled by dbm_stem_fwd_flat) -> a3 (n, 64, H, W) fp32 NCHW."""
        n, H, W = self.n, self.H, self.W
        st = ops.stream()
        ops.call("dbm_flat_conv3x3_chain", self.table.ctypes.data, self.table_dev.data_ptr(), len(self.table), n, H, W,
                 0, 0, self.flags.data_ptr(), st)
        a3 = ops.empty(n, 64, H, W)
        ops.call("dbm_flat_to_nchw", self.a3f.data_ptr(), None, a3.data_ptr(), 64, n, H, W, st)
        return a3


# ---- single-layer helpers (tests, diagnostics) -----------------------------------------------------
def pack_dgrad(w: torch.Tensor) -> torch.Tensor:
    """Data-gradient operand image of an fp32 (O, Cin, 3, 3) filter: GEMM N = Cin, K = O, taps flipped."""
    from .model import PACK_ENTRY_DTYPE
    o, cin = int(w.shape[0]), int(w.shape[1])
    out = ops.empty(9 * cin * o, dtype=torch.bfloat16)
    table = np.array([(w.data_ptr(), out.data_ptr(), cin, 0, o, cin, 0, cin, 16, 1)], dtype=PACK_ENTRY_DTYPE)
    tdev = torch.from_numpy(table.view(np.uint8).copy()).cuda()
    ops.call("dbm_pack_conv3x3_table", tdev.data_ptr(), 1, 9 * cin * o, ops.stream())
    torch.cuda.current_stream().synchronize()   # tdev must outlive the launch
    return out


def alloc_bf16(c: int, geom: dict) -> torch.Tensor:
    return torch.zeros(c // 8, geom["Pg"], 8, dtype=torch.bfloat16, device="cuda")


def alloc_f32(c: int, geom: dict) -> torch.Tensor:
    return torch.zeros(c // 4, geom["Pg"], 4, dtype=torch.float32, device="cuda")


def from_nchw(src: torch.Tensor, dst8=None, dst4=None, scale: float = 1.0):
    n, c, h, w = src.shape
    ops.call("dbm_flat_from_nchw", src.data_ptr(), c, dst8.data_ptr() if dst8 is not None else None,
             dst4.data_ptr() if dst4 is not None else None, float(scale), n, h, w, ops.stream())


def to_nchw(src: torch.Tensor, c: int, n: int, h: int, w: int, c0: int = 0) -> torch.Tensor:
    """Channels [c0, c0 + c) of a flat slab4 (fp32) or slab8 (bf16) buffer -> (n, c, h, w) fp32."""
    dst = ops.empty(n, c, h, w)
    pg = src.shape[1]
    if src.dtype == torch.float32:
        ops.call("dbm_flat_to_nchw", src.data_ptr() + 4 * c0 * pg, None, dst.data_ptr(), c, n, h, w, ops.stream())
    else:
        ops.call("dbm_flat_to_nchw", None, src.data_ptr() + 2 * c0 * pg, dst.data_ptr(), c, n, h, w, ops.stream())
    return dst


def conv3x3(inp: torch.Tensor, cin: int, wpacked: torch.Tensor, nout: int, blocks, n: int, h: int, w: int, c0: int = 0):
    """One flat 3x3 conv launch; ``blocks`` = list of dicts of FlatEpiBlock fields (device addresses)."""
    L = np.zeros(1, dtype=LAUNCH_DTYPE)
    L[0]["in"] = inp.data_ptr() + 2 * c0 * inp.shape[1]
    L[0]["wpacked"] = wpacked.data_ptr()
    L[0]["cin"] = cin
    L[0]["nout"] = nout
    L[0]["ny"] = 1
    for b, kw in enumerate(blocks):
        L[0]["blk"][b] = epi(**kw)
    ops.call("dbm_flat_conv3x3_seq", L.ctypes.data, 1, n, h, w, 0, 0, ops.stream())


# ====================================================================================================
# Single convolutions on the flat tensor-core kernels (discriminator, generator head)
# ====================================================================================================
def _round_up(a: int, b: int) -> int:
    return (a + b - 1) // b * b


class ConvImages:
    """bf16 operand images of ONE convolution's filter for the flat kernels: forward images (one per chunk of
    <= 128 output channels) and data-gradient images (one per chunk of <= 128 input / phase channels).
    ksize 3 (stride 1, pad 1) or ksize 4 (stride 2, pad 1: embedded as 3x3 over the 4 space-to-depth phases,
    PackEntry modes 2 / 3). ``entries`` are PackEntry records for dbm_pack_conv3x3_table."""

    def __init__(self, w: torch.Tensor, bias=None):
        O, C, k, k2 = (int(v) for v in w.shape)
        if (k, k2) not in ((3, 3), (4, 4)):
            raise ValueError("flat convolutions implement 3x3 stride-1 and 4x4 stride-2 filters")
        self.O, self.C, self.k = O, C, k
        self.s2d = k == 4
        self.Cg = 4 * C if self.s2d else C
        if self.Cg % 16:
            raise ValueError(f"flat convolution needs a multiple of 16 GEMM input channels, got {self.Cg}")
        self.Opad = _round_up(O, 32)
        self.Nf = min(self.Opad, 128)
        self.ny_f = self.Opad // self.Nf
        self.Nd = min(self.Cg, 128)
        self.ny_d = self.Cg // self.Nd
        assert self.Opad % self.Nf == 0 and self.Cg % self.Nd == 0 and self.Nd % 32 == 0
        bf = torch.bfloat16
        self.fwd_img = ops.zeros(self.ny_f, 9 * self.Cg * self.Nf, dtype=bf)
        self.dgrad_img = ops.zeros(self.ny_d, 9 * self.Opad * self.Nd, dtype=bf)
        self.bias = bias
        self.bias_pad = None
        if bias is not None:
            self.bias_pad = bias if self.Opad == O else ops.zeros(self.Opad)
        kk = k * k
        self.entries = []
        for y in range(self.ny_f):
            rows = min(self.Nf, O - y * self.Nf)
            self.entries.append((w.data_ptr() + 4 * y * self.Nf * C * kk, self.fwd_img[y].data_ptr(), rows, 0, self.Cg, C, 0,
                                 self.Nf, 16, 2 if self.s2d else 0))
        for y in range(self.ny_d):
            self.entries.append((w.data_ptr(), self.dgrad_img[y].data_ptr(), self.Nd, O if O < self.Opad else 0,
                                 self.Opad, C, y * self.Nd, self.Nd, 16, 3 if self.s2d else 1))
        self.max_elements = max(9 * self.Cg * self.Nf, 9 * self.Opad * self.Nd)

    def refresh_bias(self):
        if self.bias_pad is not None and self.bias_pad is not self.bias:
            self.bias_pad[: self.O].copy_(self.bias)


def pack_images(images, table=None):
    """One table-driven launch (re)packing the operand images of every ConvImages in ``images``. Returns the device
    table; pass it back in on later calls (the entries only hold pointers, which do not change)."""
    from .model import PACK_ENTRY_DTYPE
    n_entries = sum(len(im.entries) for im in images)
    if table is None:
        entries = [e for im in images for e in im.entries]
        table = torch.from_numpy(np.array(entries, dtype=PACK_ENTRY_DTYPE).view(np.uint8).copy()).cuda()
    ops.call("dbm_pack_conv3x3_table", table.data_ptr(), n_entries, max(im.max_elements for im in images),
             ops.stream())
    for im in images:
        im.refresh_bias()
    return table   # keep alive until the launch has run (callers cache it)


class FlatConv:
    """Forward / backward of one convolution for a fixed (batch, H, W), NCHW fp32 tensors in and out, on the flat
    tcgen05 kernels (bf16 operands, fp32 accumulation). ``nslots`` forward inputs can be kept for backward (the
    discriminator step runs two forward passes before its two backward passes, srgan_train.py:1145-1163)."""

    TARGET_UNITS = 296

    def __init__(self, im: ConvImages, gw: torch.Tensor, n: int, H: int, W: int, act: bool = False, nslots: int = 1):
        self.im, self.n, self.H, self.W, self.act = im, n, H, W, act
        s2d = im.s2d
        self.Ho, self.Wo = (H // 2, W // 2) if s2d else (H, W)
        self.gh, self.gw_ = ((H + 1) // 2, (W + 1) // 2) if s2d else (H, W)
        if self.Ho < 1 or self.Wo < 1:
            raise ValueError("input too small for this convolution")
        self.geom = geometry(n, self.gh, self.gw_)
        Pg = self.geom["Pg"]
        self.Pg = Pg
        self.xin = [alloc_bf16(im.Cg, self.geom) for _ in range(nslots)]
        self.zf = alloc_f32(im.Opad, self.geom)
        self.gin = alloc_bf16(im.Opad, self.geom)
        self.dxf = alloc_f32(im.Cg, self.geom)
        self.rec_f = []
        for slot in range(nslots):
            L = np.zeros(1, dtype=LAUNCH_DTYPE)
            L[0]["in"] = self.xin[slot].data_ptr()
            L[0]["wpacked"] = im.fwd_img.data_ptr()
            L[0]["cin"], L[0]["nout"], L[0]["ny"] = im.Cg, im.Nf, im.ny_f
            L[0]["w_chunk_stride"] = 9 * im.Cg * im.Nf
            for b in range(im.Nf // 32):
                L[0]["blk"][b] = epi(bias=(im.bias_pad.data_ptr() + 128 * b) if im.bias_pad is not None else 0,
                                     act=int(act), out_f32=self.zf.data_ptr() + 4 * 32 * b * Pg)
            self.rec_f.append(L)
        L = np.zeros(1, dtype=LAUNCH_DTYPE)
        L[0]["in"] = self.gin.data_ptr()
        L[0]["wpacked"] = im.dgrad_img.data_ptr()
        L[0]["cin"], L[0]["nout"], L[0]["ny"] = im.Opad, im.Nd, im.ny_d
        L[0]["w_chunk_stride"] = 9 * im.Opad * im.Nd
        for b in range(im.Nd // 32):
            L[0]["blk"][b] = epi(out_f32=self.dxf.data_ptr() + 4 * 32 * b * Pg)
        self.rec_d = L
        # weight gradient: units = (input-channel chunk, 32 output channels, position range)
        chunks = chunk_channels(im.Cg)
        ogroups = im.Opad // 32
        nsplit = max(1, min(self.geom["tiles"], round(self.TARGET_UNITS / (len(chunks) * ogroups))))
        splits = split_blocks(self.geom["tiles"], nsplit)
        self.units, self.n_units = [], 0
        reduces = []
        dev = lambda a: torch.from_numpy(a.view(np.uint8).reshape(-1).copy()).cuda()
        n_units = len(chunks) * ogroups * len(splits)
        self.partial = torch.empty(n_units * PARTIAL_FLOATS, dtype=torch.float32, device="cuda")
        base = self.partial.data_ptr()
        for slot in range(nslots):
            units = []
            for og in range(ogroups):
                for c0, nch in chunks:
                    first = len(units)
                    for blk0, nblk in splits:
                        units.append((self.xin[slot].data_ptr() + 2 * c0 * Pg, self.gin.data_ptr() + 2 * 32 * og * Pg,
                                      base + len(units) * PARTIAL_FLOATS * 4, blk0, nblk, nch // 8,
                                      s2d_tap_mask(c0, nch, im.C) if s2d else 0, (0, 0)))
                    if slot == 0:
                        ovalid = min(32, im.O - 32 * og)
                        mode = (1 if s2d else 0) | ((ovalid if ovalid < 32 else 0) << 8)
                        reduces.append((base + first * PARTIAL_FLOATS * 4, gw.data_ptr(), PARTIAL_FLOATS, len(splits), im.C,
                                        c0, 32 * og, nch, mode))
            self.units.append(dev(np.array(units, dtype=WGRAD_UNIT_DTYPE)))
            self.n_units = len(units)
        self.reduce_dev, self.n_reduce = dev(np.array(reduces, dtype=WGRAD_REDUCE_DTYPE)), len(reduces)
        self.flops = 2.0 * 9 * im.Cg * im.Opad * self.geom["P"]   # executed MMA FLOPs per GEMM pass

    def forward(self, x: torch.Tensor, slot: int = 0) -> torch.Tensor:
        im, n, st = self.im, self.n, ops.stream()
        ops.call("dbm_flat_from_nchw_ex", x.data_ptr(), im.C, self.H, self.W, int(im.s2d), self.xin[slot].data_ptr(), None,
                 1.0, n, self.gh, self.gw_, st)
        ops.call("dbm_flat_conv3x3_seq", self.rec_f[slot].ctypes.data, 1, n, self.gh, self.gw_, self.Ho, self.Wo, st)
        z = ops.empty(n, im.O, self.Ho, self.Wo)
        ops.call("dbm_flat_to_nchw_ex", self.zf.data_ptr(), None, z.data_ptr(), im.O, self.Ho, self.Wo, 0, n, self.gh,
                 self.gw_, st)
        return z

    def backward(self, dz: torch.Tensor, slot: int = 0, need_dx: bool = True, wgrad_stream=None):
        """dW += x (*) dz for the input kept in ``slot``; returns d(loss)/dx (n, C, H, W) or None.
        ``wgrad_stream``: torch stream for the weight-gradient launches (nothing downstream in backward needs them: they
        run beside the data-gradient chain; the CALLER joins that stream before using the gradients)."""
        im, n, st = self.im, self.n, ops.stream()
        ops.call("dbm_flat_from_nchw_ex", dz.data_ptr(), im.O, self.Ho, self.Wo, 0, self.gin.data_ptr(), None, 1.0, n,
                 self.gh, self.gw_, st)
        if wgrad_stream is not None:
            wgrad_stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(wgrad_stream):
                ws = ops.stream()
                ops.call("dbm_flat_wgrad", self.units[slot].data_ptr(), self.n_units, n, self.gh, self.gw_, ws)
                ops.call("dbm_flat_wgrad_reduce", self.reduce_dev.data_ptr(), self.n_reduce, ws)
        dx = None
        if need_dx:
            ops.call("dbm_flat_conv3x3_seq", self.rec_d.ctypes.data, 1, n, self.gh, self.gw_, 0, 0, st)
            dx = ops.empty(n, im.C, self.H, self.W)
            ops.call("dbm_flat_to_nchw_ex", self.dxf.data_ptr(), None, dx.data_ptr(), im.C, self.H, self.W, int(im.s2d), n,
                     self.gh, self.gw_, st)
        if wgrad_stream is None:
            ops.call("dbm_flat_wgrad", self.units[slot].data_ptr(), self.n_units, n, self.gh, self.gw_, st)
            ops.call("dbm_flat_wgrad_reduce", self.reduce_dev.data_ptr(), self.n_reduce, st)
        return dx
