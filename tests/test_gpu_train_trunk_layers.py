"""Pass-by-pass value checks of the tensor-core TRAINING trunk (deepbedmap_b200/flat.py: the image-resident kernels of
csrc/umma_local.cu, the flat layer chain, the batched weight gradient and the bias gradient of csrc/umma_flat.cu), each
against float64 on the buffers the kernels read, exactly as stored.

Model-level parity cannot see a wrong backward pass: every dense-block gradient reaches d(a0) scaled by beta * sigma,
and a relative L2 over the whole gradient vector dilutes a defect in one of 36 blocks. Here one training step runs as
shipped (forward, then backward with the weight gradients on a side stream, into a pre-filled ``flat_grad``), and then
  * every kept activation a_k of every dense block j is recomputed from cat[j][:64 + G (k - 1)] as stored;
  * the data-gradient chain is teacher-forced: inside a block, each gradient slot g_{k-1} is recomputed from the
    kernel's own stored g_k .. g_5 and the LeakyReLU derivative of the stored bf16 activation (0.2 where its sign bit is
    set); across blocks the fp32 gradient stream dX_j is carried in float64 from the kernel's stored gradients:
        dX_nrdb = D_post(gpost),  dX_j = D_a0(block j) + sigma_j dX_{j+1} + [r = 1] dX_{j+3} + [j = 0] da3
    and every block's g5 = bf16(beta sigma_j dX_{j+1}), gpre and d(a0) are checked against it;
  * every trunk parameter's weight and bias gradient is recomputed from its (activation, gradient) pair;
  * where the fp32 residual or gradient stream is exposed (the flat chain's rings after prefix runs of its launch
    table, the image-resident kernel's scratch after prefixes of its pass table) it is compared on its branch, with the
    skip terms removed.
The references follow the model's equations (oracle.residual_dense_block / rrdb / trunk_forward, srgan_train.py:339-358,
397-402, 541-551): sigma_j = beta for the third block of an RRDB (its output is scaled again, :402), 1 otherwise. The
filters are the bf16 rounding of the fp32 master weights, never the packed operand images. The flat buffers are read
through plain torch views of their layout ([C/8][Pg][8] bf16, [C/4][Pg][4] fp32; image i's padded position
G0 + i (H+2)(W+2) + y (W+2) + x), not through the library's own layout kernels.

Bounds: see layer_check.py. Outputs compared on a branch add the fp32 rounding of the kernel's skip additions, divided
by the branch's scale. A CPU test checks the reference recursion itself against autograd of the oracle's trunk, and a
self-test feeds every comparison deliberately wrong references, each of which must fail.

Run with -s to see, per (pass kind, output kind) and configuration, the worst element error / bound and relative L2.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import deepbedmap_oracle as O
from layer_check import F64, TOL_REL, Report, bound_of, ulp_bf16, ulp_f32

SLOPE = float(np.float32(0.2))       # kLreluSlope
BETA = 0.1
TRUNK = ("pre_residual_conv_layer/", "residual_network/", "post_residual_conv_layer/")
PRE, POST = "pre_residual_conv_layer", "post_residual_conv_layer"


def block_key(j, k):
    """Parameter prefix of conv_k of residual dense block j (0-based over the whole trunk, three per RRDB)."""
    return f"residual_network/{j // 3}/residual_dense_block{j % 3 + 1}/conv_layer{k}"


def key_block(key):
    """block_key inverse: (j, k), or None for the pre- / post-residual conv."""
    if not key.startswith("residual_network/"):
        return None
    _, i, rdb, conv = key.split("/")
    return 3 * int(i) + int(rdb[len("residual_dense_block"):]) - 1, int(conv[len("conv_layer"):])


def pad(t):
    return F.pad(t, (1, 1, 1, 1))


def inner(t):
    return t[..., 1:-1, 1:-1]


# ---- the model's equations in float64 on padded NCHW tensors ---------------------------------------------------------
class Equations:
    """Convolutions of the trunk (3x3, padding 1) on (n, C, H + 2, W + 2) tensors whose border is the stored one.
    ``w`` / ``b``: float64 filters and biases by parameter prefix. Each op returns (value, S), S the same contraction of
    the operands' magnitudes. ``defect`` plants a deliberately wrong reference (checker self-test)."""

    def __init__(self, w, b, nb, G, beta, slope, defect=None):
        self.w, self.b, self.nb, self.G, self.beta, self.slope = w, b, nb, G, beta, slope
        self.nrdb, self.cc = 3 * nb, 64 + 4 * G
        self.defect = defect or {}

    def lrelu(self, v):
        return torch.where(v >= 0, v, self.slope * v)

    def mask(self, a):
        """LeakyReLU derivative, defined by the sign bit of the stored activation."""
        m = torch.ones_like(a, dtype=F64)
        m[torch.signbit(a)] = self.slope
        return m

    def sigma(self, j):
        """d(x_{j+1}) / d(x_j) through the skip of block j: beta when block j closes an RRDB (:402), else 1."""
        return self.defect.get("sigma", {}).get(j, self.beta if j % 3 == 2 else 1.0)

    def fwd(self, x, key):
        w = self.w[key]
        x = x[:, :w.shape[1]]
        return F.conv2d(x, w) + self.b[key].view(1, -1, 1, 1), F.conv2d(x.abs(), w.abs())

    def dgrad(self, g, key, jk=None):
        """d(loss)/d(input) of conv ``key`` from its padded output gradient g: (n, cin, H, W)."""
        w = self.w[key]
        fix = self.defect.get("dgrad_w", {}).get(jk)
        if fix is not None:
            w = fix(w.clone())
        wt = w.flip(2, 3).transpose(0, 1)
        return F.conv2d(g, wt), F.conv2d(g.abs(), wt.abs())

    def wgrad(self, a, g):
        """dW (cout, cin, 3, 3) = sum over images and pixels of g (interior) x a (padded), and db."""
        dw = F.conv2d(a.transpose(0, 1), g.transpose(0, 1)).transpose(0, 1)
        S = F.conv2d(a.abs().transpose(0, 1), g.abs().transpose(0, 1)).transpose(0, 1)
        return dw, S, g.sum((0, 2, 3)), g.abs().sum((0, 2, 3))

    def forward_chain(self, s0):
        """Exact forward (no rounding): padded dense-block buffers cats[0..nrdb] and x_0, a3."""
        x0 = self.lrelu(self.fwd(s0, PRE)[0])
        x, cats = x0, []
        for j in range(self.nrdb):
            if j % 3 == 0:
                rrdb_in = x
            cat = pad(x)
            for k in (1, 2, 3, 4):
                cat = torch.cat([cat, pad(self.lrelu(self.fwd(cat, block_key(j, k))[0]))], 1)
            c5 = self.fwd(cat, block_key(j, 5))[0]
            x = x + self.beta * c5 if j % 3 != 2 else rrdb_in + self.beta * (x + self.beta * c5)   # :358, :402
            cats.append(cat)
        cats.append(pad(x))
        return cats, x0, x0 + self.fwd(pad(x), POST)[0]

    def backward_chain(self, cats, gpost, da3, take, keep=False):
        """The data-gradient chain. ``take(name, j, k, ref, S)`` receives the reference of each bf16 gradient
        (g_k of block j, name "g"; g5, name "g5"; "gpre") and returns the padded gradient used downstream: the
        kernel's stored one (teacher forcing) or the reference itself. Returns the stream {j: (dX_j, S)}, the
        per-block {j: (D_a0, S)}, d(a0) with S, and (keep) every {(j, k): (D_k(g_k), S)}."""
        G, nrdb, d = self.G, self.nrdb, self.defect
        dX = {nrdb: self.dgrad(gpost, POST)}
        da0_blk, Dk = {}, {}
        for j in reversed(range(nrdb)):
            sg = self.sigma(j)
            x1, s1 = dX[j + 1]
            g = {5: take("g5", j, 5, self.beta * sg * x1, self.beta * sg * s1)}
            acc = torch.zeros_like(cats[j][:, :, 1:-1, 1:-1])
            sacc = torch.zeros_like(acc)
            for k in (5, 4, 3, 2):
                v, S = self.dgrad(g[k], block_key(j, k), (j, k))
                cin = v.shape[1]
                acc[:, :cin] += v
                sacc[:, :cin] += S
                if keep:
                    Dk[(j, k)] = (v, S)
                slot = slice(cin - G, cin)                     # slot a_{k-1} is final after conv_k's gradient
                mk = self.mask(inner(cats[j][:, slot]))
                if d.get("mask_off") == (j, k - 1):
                    mk = torch.ones_like(mk)
                g[k - 1] = take("g", j, k - 1, mk * acc[:, slot], mk * sacc[:, slot])
            v, S = self.dgrad(g[1], block_key(j, 1), (j, 1))
            if keep:
                Dk[(j, 1)] = (v, S)
            da0, sda0 = acc[:, :64] + v, sacc[:, :64] + S
            da0_blk[j] = (da0, sda0)
            x, s = da0 + sg * x1, sda0 + sg * s1
            if j % 3 == 0 and j + 3 <= nrdb and j not in d.get("no_rrdb_skip", ()):
                x, s = x + dX[j + 3][0], s + dX[j + 3][1]       # x_{j+3} = x_j + beta * (...) (:402)
            if j == 0:
                x, s = x + da3, s + da3.abs()                   # a3 = a1 + post_res(...) (:551)
            dX[j] = (x, s)
        mk = self.mask(inner(cats[0][:, :64]))
        gpre = take("gpre", 0, 0, mk * dX[0][0], mk * dX[0][1])
        return dX, da0_blk, self.dgrad(gpre, PRE), Dk

    def conv_pairs(self, s0, cats, gslot, gpre, gpost):
        """(parameter prefix, activation, output gradient) of every trunk conv: 2 + 15 nb pairs."""
        G = self.G
        out = [(PRE, s0, gpre)]
        for j in range(self.nrdb):
            for k in (1, 2, 3, 4, 5):
                out.append((block_key(j, k), cats[j][:, :64 + G * (k - 1)] if k < 5 else cats[j], gslot(j, k)))
        out.append((POST, cats[self.nrdb][:, :64], gpost))
        return out


# ---- flat-layout views -------------------------------------------------------------------------------------------------
class Layout:
    def __init__(self, geom, n, H, W):
        self.n, self.H, self.W, self.G0, self.Pg = n, H, W, geom["G0"], geom["Pg"]
        self.Hp, self.Wp = H + 2, W + 2
        self.P = n * self.Hp * self.Wp
        interior = torch.zeros(self.Pg, dtype=torch.bool, device="cuda")
        interior[self.G0:self.G0 + self.P].view(n, self.Hp, self.Wp)[:, 1:H + 1, 1:W + 1] = True
        self.border = ~interior

    def padded(self, t):
        """[C/v][Pg][v] flat buffer -> (n, C, H + 2, W + 2) float64, borders as stored."""
        cs, _, v = t.shape
        x = t[:, self.G0:self.G0 + self.P].reshape(cs, self.n, self.Hp, self.Wp, v)
        return x.permute(1, 0, 4, 2, 3).reshape(self.n, cs * v, self.Hp, self.Wp).to(F64)

    def scratch(self, t):
        """x_scratch row of the image-resident kernel, [n][16][128][4] fp32 at m = y (W+2) + x -> (n, 64, H, W)."""
        x = t.view(self.n, 16, 128, 4)[:, :, :self.Hp * self.Wp].reshape(self.n, 16, self.Hp, self.Wp, 4)
        return inner(x.permute(0, 1, 4, 2, 3).reshape(self.n, 64, self.Hp, self.Wp)).to(F64)

    def check_borders(self, rep, label, t):
        """Every border and guard position of a flat buffer is exactly zero."""
        rep.exact(label + " borders", t[:, self.border], torch.zeros_like(t[:, self.border]))


def fp32_branch(rep, label, got, skip, ref, S, slack):
    """fp32 result compared on its branch: got - skip against ref, plus the fp32 rounding of the skip additions. The
    relative-L2 cap grows by the same rounding in that norm: where the branch is small beside the skip (the dense
    block accumulator dcat after conv2 .. conv4's gradients) half an fp32 ulp of the sum is ~1e-5 of the branch."""
    cap = TOL_REL["f32"] + float(torch.as_tensor(slack).broadcast_to(ref.shape).norm() / ref.norm().clamp_min(1e-300))
    rep.add(label, "f32", got - skip, ref, bound_of("f32", ref, S) + slack, rel_limit=cap)


def half_ulp(*ts):
    return sum(0.5 * ulp_f32(t) for t in ts)


# ---- one training step of the trunk, as shipped ------------------------------------------------------------------------
def make_model(nb, G, seed=0):
    from deepbedmap_b200 import GeneratorModel
    params = O.init_generator_params(nb, seed=seed, bias_std=0.1, scale=0.7, inter_channels=G)
    m = GeneratorModel(num_residual_blocks=nb, residual_scaling=BETA, inter_channels=G)
    assert m.train_precision == "bf16"
    for k, v in params.items():
        m.set_param(k, v)
    return m


class TrainStep:
    def __init__(self, nb, G, n, H, W, local, seed=0):
        from deepbedmap_b200 import flat, ops
        self.flat, self.ops = flat, ops
        self.m = m = make_model(nb, G, seed)
        self.nb, self.G, self.n, self.H, self.W, self.nrdb = nb, G, n, H, W, 3 * nb
        self.ft = ft = m._flat_trunk(n, H, W)
        assert ft.local_dev is not None or not local, "the image-resident kernel does not apply to this shape"
        ft.local = local
        self.lay = Layout(ft.geom, n, H, W)
        g = torch.Generator(device="cuda").manual_seed(100 + seed)
        self.a0 = torch.randn(n, 128, H, W, generator=g, device="cuda")
        self.da3 = torch.randn(n, 64, H, W, generator=g, device="cuda")
        # accumulation is part of the contract: the step adds onto whatever flat_grad holds
        self.prefill = torch.randn(m.flat_grad.numel(), generator=g, device="cuda") * 0.01
        self.side = torch.cuda.Stream()
        q = lambda t: t.bfloat16().to(F64)
        self.eq_w = {k[:-2]: q(v) for k, v in m.p.items() if k.startswith(TRUNK) and k.endswith("/W")}
        self.eq_b = {k[:-2]: v.to(F64) for k, v in m.p.items() if k.startswith(TRUNK) and k.endswith("/b")}

    def equations(self, defect=None):
        return Equations(self.eq_w, self.eq_b, self.nb, self.G, BETA, SLOPE, defect)

    def run(self):
        ft = self.ft
        self.m.flat_grad.copy_(self.prefill)
        ft.forward(self.a0)
        ft.backward(self.da3, wgrad_stream=self.side)
        torch.cuda.synchronize()
        snap = dict(s0=ft.s0, cat=ft.cat, gcat=ft.gcat, gpost=ft.gpost, gpre=ft.gpre, da3f=ft.da3f, da0f=ft.da0f,
                    a3f=ft.a3f, grad=self.m.flat_grad)
        snap["x0"] = ft.x_scratch[0] if ft.local else ft.x0
        return {k: [t.clone() for t in v] if isinstance(v, list) else v.clone() for k, v in snap.items()}

    def grad_of(self, flat, key):
        o, cnt = self.m._slices[key]
        return flat[o:o + cnt].view(self.m.p[key].shape)

    # -- items 1-4: the final state of the step --
    def check(self, snap, rep, defect=None):
        eq, lay, G, nrdb = self.equations(defect), self.lay, self.G, self.nrdb
        d = defect or {}
        cats = [lay.padded(c) for c in snap["cat"]]
        gcats = [lay.padded(c) for c in snap["gcat"]]
        s0, gpost, gpre = lay.padded(snap["s0"]), lay.padded(snap["gpost"]), lay.padded(snap["gpre"])
        # kept forward activations
        self.c5 = {}
        for j in range(nrdb):
            for k in (1, 2, 3, 4):
                cin = 64 + G * (k - 1)
                y, S = eq.fwd(cats[j], block_key(j, k))
                ref = eq.lrelu(y)
                rep.add(f"a{k} (fwd conv{k})", "bf16", inner(cats[j][:, cin:cin + G]), ref, bound_of("bf16", ref, S))
            self.c5[j] = eq.fwd(cats[j], block_key(j, 5))
        x0 = lay.scratch(snap["x0"]) if self.ft.local else inner(lay.padded(snap["x0"]))
        y, S = eq.fwd(s0, PRE)
        ref = eq.lrelu(y)
        rep.add("x0 (fwd pre-residual)", "f32", x0, ref, bound_of("f32", ref, S))
        rep.exact("x0 bf16 copy", inner(snap_bf16(snap["cat"][0], lay))[:, :64], x0.float().bfloat16())
        a3f = inner(lay.padded(snap["a3f"]))
        y, S = eq.fwd(cats[nrdb], POST)
        fp32_branch(rep, "a3 - x0 (fwd post-residual)", a3f, x0, y, S, half_ulp(a3f))
        # data-gradient chain, teacher-forced on the stored gradients
        da3 = inner(lay.padded(snap["da3f"]))
        rep.exact("da3 bf16 copy", inner(snap_bf16(snap["gpost"], lay)), da3.float().bfloat16())

        def stored(name, j, k):
            if name == "gpre":
                return gpre[:, :64]
            return gcats[j][:, G * (k - 1):G * k] if k < 5 else gcats[j][:, 4 * G:4 * G + 64]

        def take(name, j, k, ref, S):
            if "g_fix" in d:
                ref = d["g_fix"](name, j, k, ref)
            got = stored(name, j, k)
            label = {"g": f"g{k} (dgrad conv{k + 1}..5)", "g5": "g5 (dX_j+1 stream)", "gpre": "gpre (dX_0 stream)"}[name]
            rep.add(label, "bf16", inner(got), ref, bound_of("bf16", ref, S))
            return got

        dX, da0_blk, (da0, S), self.Dk = eq.backward_chain(cats, gpost, da3, take, keep=not self.ft.local)
        self.dX, self.da0_blk = dX, da0_blk
        rep.add("d(a0) (dgrad pre-residual)", "f32", inner(lay.padded(snap["da0f"])), da0, bound_of("f32", da0, S))
        # weight and bias gradients, each trunk parameter on its own
        pairs = eq.conv_pairs(s0, cats, lambda j, k: stored("g", j, k) if k < 5 else stored("g5", j, 5), gpre[:, :64],
                              gpost)
        assert len(pairs) == 2 + 15 * self.nb
        for key, a, g in pairs:
            g = inner(g)
            if key in d.get("wgrad_positions", {}):
                g = g * d["wgrad_positions"][key]
            dw, Sw, db, Sb = eq.wgrad(a, g)
            if key in d.get("wgrad_fix", {}):
                dw = d["wgrad_fix"][key](dw.clone())
            kind = key.rsplit("/", 1)[-1]
            for suffix, ref, S in (("W", dw, Sw), ("b", db, Sb)):
                tot = self.grad_of(snap["grad"], f"{key}/{suffix}").to(F64)
                got = tot - self.grad_of(self.prefill, f"{key}/{suffix}").to(F64)
                rep.add(f"d{suffix} {kind}", "f32", got, ref, bound_of("f32", ref, S) + half_ulp(tot))
        for key in self.m.p:
            if not key.startswith(TRUNK):
                rep.exact("untouched non-trunk gradients", self.grad_of(snap["grad"], key).view(torch.int32),
                          self.grad_of(self.prefill, key).view(torch.int32))
        # layout: the weight / bias gradients sum over every flat position, borders included
        for name in ("s0", "gpost", "gpre"):
            lay.check_borders(rep, name, snap[name])
        for t in (d["border_fix"](snap["cat"]) if "border_fix" in d else snap["cat"]):
            lay.check_borders(rep, "cat", t)
        for t in snap["gcat"]:
            lay.check_borders(rep, "gcat", t)

    def check_rerun(self, snap, rep):
        """A second step from the same inputs and pre-filled gradients gives the same bits."""
        again = self.run()
        for k, v in snap.items():
            for i, (a, b) in enumerate(zip(v, again[k]) if isinstance(v, list) else [(v, again[k])]):
                rep.exact(f"second step: {k}", a.view(torch.int16) if a.dtype == torch.bfloat16 else a.view(torch.int32),
                          b.view(torch.int16) if b.dtype == torch.bfloat16 else b.view(torch.int32))

    # -- the exposed fp32 streams, after prefix runs --
    def check_local_prefixes(self, rep):
        """x_scratch of the image-resident kernel: the RRDB input stream after forward prefixes ending at an RRDB end,
        the gradient stream of the RRDB in front after backward prefixes ending at an r = 1 block (j > 0)."""
        from deepbedmap_b200 import flat
        ft, lay, eq, ops, nrdb = self.ft, self.lay, self.equations(), self.ops, self.nrdb
        n, H, W, st = self.n, self.H, self.W, ops.stream()
        cat = lambda j: snap_bf16(ft.cat[j], lay)
        tab = np.frombuffer(ft.local_dev.cpu().numpy().tobytes(), dtype=flat.LOCAL_PASS_DTYPE)
        ends = [i for i, r in enumerate(tab) if int(r["type"]) == flat.LOC_RDB and int(r["rr"])]
        assert len(ends) == self.nb and len(tab) == 2 + 5 * nrdb
        x_prev = lay.scratch(ft.x_scratch[0])            # x_0 (checked against the reference in check())
        for i, e in enumerate(ends):
            j = 3 * i + 2
            ft.x_scratch[1].fill_(float("nan"))
            ops.call("dbm_trunk_local_fwd", ft.local_dev.data_ptr(), e + 1, n, H, W, ft.s0.data_ptr(),
                     ft.x_scratch[0].data_ptr(), ft.x_scratch[1].data_ptr(), st)
            torch.cuda.synchronize()
            x = lay.scratch(ft.x_scratch[1])
            # x_{j+1} = x_{j-2} + beta (x_j + beta c5_j), x_j = x_{j-2} + beta (c5_{j-2} + c5_{j-1}) (:358, :402)
            (ca, sa), (cb, sb), (cc_, sc) = self.c5[j - 2], self.c5[j - 1], self.c5[j]
            x1 = x_prev + BETA * ca
            x2 = x1 + BETA * cb
            t = x2 + BETA * cc_
            slack = (half_ulp(x) + BETA * half_ulp(t, x2, x1)) / BETA ** 2 + half_ulp(ca, cb, cc_)
            fp32_branch(rep, "x RRDB out (image-resident fwd)", (x - (1 + BETA) * x_prev) / BETA ** 2, 0.0,
                        ca + cb + cc_, sa + sb + sc, slack)
            rep.exact("x RRDB out bf16 copy", inner(cat(j + 1))[:, :64], x.float().bfloat16())
            x_prev = x
        tab = np.frombuffer(ft.local_bwd_dev.cpu().numpy().tobytes(), dtype=flat.LOCAL_PASS_DTYPE)
        d1 = [i for i, r in enumerate(tab) if int(r["type"]) == flat.LOC_BD1]   # conv1 of blocks nrdb - 1 .. 0
        assert len(d1) == nrdb and len(tab) == 2 + 5 * nrdb
        gpost = ft.gpost.data_ptr()
        dx_next = None
        for count, j in [(1, nrdb)] + [(d1[nrdb - 1 - j] + 1, j) for j in reversed(range(3, nrdb, 3))]:
            ft.x_scratch[1].fill_(float("nan"))
            ops.call("dbm_trunk_local_bwd", ft.local_bwd_dev.data_ptr(), count, n, H, W, gpost,
                     ft.x_scratch[1].data_ptr(), st)
            torch.cuda.synchronize()
            dx = lay.scratch(ft.x_scratch[1])
            if j == nrdb:
                ref, S = self.dX[nrdb]
                rep.add("dX_nrdb (image-resident dgrad post)", "f32", dx, ref, bound_of("f32", ref, S))
            else:
                # dX_j = D_j + D_{j+1} + D_{j+2} + (1 + beta) dX_{j+3} over one RRDB (:358, :402)
                (da, sa), (db_, sb), (dc, sc) = (self.da0_blk[j + i] for i in range(3))
                y2 = dc + BETA * dx_next
                y1 = db_ + y2
                slack = half_ulp(y2, y1, da + y1, dx)
                fp32_branch(rep, "dX RRDB in (image-resident dgrad)", dx, (1 + BETA) * dx_next, da + db_ + dc,
                            sa + sb + sc, slack)
            dx_next = dx

    def check_chain_prefixes(self, rep):
        """The flat chain's x ring after prefixes of the forward table ending at each block's conv5, and its dcat /
        dX ring after every prefix of the data-gradient table (each N-slice launch on its own)."""
        ft, lay, ops, nrdb, G = self.ft, self.lay, self.ops, self.nrdb, self.G
        n, H, W, st = self.n, self.H, self.W, ops.stream()
        names = {}
        for k, v in self.m._packed.items():
            if k.endswith("@trunk"):
                names[v[0].data_ptr()] = (k[:-len("@trunk")], 0, None)
            elif k.endswith("@dgrad_slices"):
                for c0, wdt, img in v:
                    names[img.data_ptr()] = (k[:-len("@dgrad_slices")], c0, wdt)

        def prefix(table, count, bufs):
            for b in bufs:
                b.fill_(float("nan"))
            ops.call("dbm_flat_conv3x3_seq", table.ctypes.data, count, n, H, W, 0, 0, st)
            torch.cuda.synchronize()

        fp = lambda t: inner(lay.padded(t))
        for L, rec in enumerate(ft.fwd):
            jk = key_block(names[int(rec["wpacked"])][0])
            if jk is None or jk[1] != 5:
                continue
            j = jk[0]
            prefix(ft.fwd, L + 1, ft.xring)
            x1, x = fp(ft._x(j + 1)), fp(ft._x(j))
            c5, S = self.c5[j]
            if j % 3 != 2:
                fp32_branch(rep, "x_j+1 (flat fwd conv5)", (x1 - x) / BETA, 0.0, c5, S, half_ulp(x1) / BETA)
            else:
                xr = fp(ft._x(j - 2))
                t = (x1 - xr) / BETA
                fp32_branch(rep, "x_j+1 RRDB out (flat fwd conv5)", (t - x) / BETA, 0.0, c5, S,
                            (half_ulp(x1) + BETA * half_ulp(t)) / BETA ** 2)
            rep.exact("x_j+1 bf16 copy", inner(snap_bf16(ft.cat[j + 1], lay))[:, :64], x1.float().bfloat16())
        da3 = fp(ft.da3f)
        prev = None
        nsliced = 0
        for L, rec in enumerate(ft.bwd):
            key, c0, wdt = names[int(rec["wpacked"])]
            prefix(ft.bwd, L + 1, [ft.dcat] + ft.dX)
            cur = dict(dcat=fp(ft.dcat), dX=[fp(t) for t in ft.dX])
            jk = key_block(key)
            if key == POST:
                ref, S = self.dX[nrdb]
                rep.add("dX_nrdb (flat dgrad post)", "f32", cur["dX"][nrdb % 4], ref, bound_of("f32", ref, S))
            elif jk is not None:
                j, k = jk
                v, S = self.Dk[(j, k)]
                cin = v.shape[1]
                nsliced += wdt < cin
                hi = min(c0 + wdt, cin - G)          # the fp32 part of this slice (slot a_{k-1} is bf16, checked above)
                lab = f"dcat (flat dgrad conv{k}{', N-slice' if wdt < cin else ''})"
                if k == 5 and c0 < hi:
                    skip = torch.zeros_like(v[:, c0:hi])
                    lo64 = max(0, min(64, hi) - c0)
                    skip[:, :lo64] = self.equations().sigma(j) * cur["dX"][(j + 1) % 4][:, c0:c0 + lo64]
                    if j == 0:
                        skip[:, :lo64] += da3[:, c0:c0 + lo64]
                    got = cur["dcat"][:, c0:hi]
                    fp32_branch(rep, lab, got, skip, v[:, c0:hi], S[:, c0:hi], half_ulp(got, skip) * 2)
                elif 1 < k < 5 and c0 < hi:
                    got, before = cur["dcat"][:, c0:hi], prev["dcat"][:, c0:hi]
                    fp32_branch(rep, lab, got, before, v[:, c0:hi], S[:, c0:hi], half_ulp(got))
                elif k == 1 and j > 0:
                    got, skip = cur["dX"][j % 4], prev["dcat"][:, :64]
                    if j % 3 == 0:
                        skip = skip + cur["dX"][(j + 3) % 4]
                    fp32_branch(rep, "dX_j (flat dgrad conv1)", got, skip, v, S, half_ulp(got, skip) * 2)
            prev = cur
        assert nsliced == (4 * nrdb if G == 64 else 0)   # two slices each of conv4 and conv5 at inter_channels 64


def snap_bf16(t, lay):
    return lay.padded(t).float().bfloat16()


# ---- configurations ----------------------------------------------------------------------------------------------------
CONFIGS = [  # (nb, inter_channels, (n, H, W), image-resident)
    (12, 32, (128, 9, 9), True),     # the benchmark's generator step
    (1, 32, (None, 9, 9), True),     # SOLO form: more images than SMs
    (2, 32, (3, 6, 14), True),       # padded image exactly 128 positions
    (2, 32, (1, 9, 9), True),        # one image
    (1, 32, (2, 5, 4), True),
    (2, 32, (2, 3, 5), True),
    (2, 32, (3, 9, 9), False),       # flat chain
    (2, 32, (2, 30, 23), False),     # flat chain, several tiles per CTA
    (2, 64, (3, 9, 9), False),       # inter_channels 64: N-sliced data gradients
    (1, 64, (2, 12, 10), False),
]


def _cfg_id(c):
    nb, G, (n, H, W), local = c
    return f"{'local' if local else 'chain'}-nb{nb}-g{G}-{'solo' if n is None else n}x{H}x{W}"


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CONFIGS, ids=[_cfg_id(c) for c in CONFIGS])
def test_train_trunk_every_pass_matches_fp64(cfg):
    nb, G, (n, H, W), local = cfg
    if n is None:
        n = torch.cuda.get_device_properties(0).multi_processor_count + 1
    step = TrainStep(nb, G, n, H, W, local)
    snap = step.run()
    rep = Report(_cfg_id(cfg))
    step.check(snap, rep)
    step.check_rerun(snap, rep)
    if local:
        step.check_local_prefixes(rep)
    else:
        step.check_chain_prefixes(rep)
    rep.finish()


# ---- the reference recursion itself (CPU) -------------------------------------------------------------------------------
def test_reference_recursion_matches_oracle_autograd():
    """Without any rounding, the reference recursion used above (the stream dX_j with sigma_j, the g5 scale beta sigma_j,
    the RRDB and a3 skips, the masks, the weight-gradient pairs) equals float64 autograd of oracle.trunk_forward, for
    d(a0) and every trunk parameter's gradient. Needs no GPU."""
    nb, G, n, H, W = 2, 32, 2, 5, 4
    params = O.init_generator_params(nb, seed=3, bias_std=0.1, scale=0.7, inter_channels=G)
    p64 = {k: torch.as_tensor(v, dtype=F64).requires_grad_(True) for k, v in params.items()}
    g = torch.Generator().manual_seed(5)
    a0 = torch.randn(n, 128, H, W, generator=g, dtype=F64).requires_grad_(True)
    da3 = torch.randn(n, 64, H, W, generator=g, dtype=F64)
    a3r = O.trunk_forward(p64, a0, nb, BETA, emulate_bf16=False)
    (a3r * da3).sum().backward()

    eq = Equations({k[:-2]: v.detach() for k, v in p64.items() if k.endswith("/W")},
                   {k[:-2]: v.detach() for k, v in p64.items() if k.endswith("/b")}, nb, G, BETA, O.LRELU_SLOPE)
    s0 = pad(a0.detach())
    cats, x0, a3 = eq.forward_chain(s0)
    kept = {}

    def take(name, j, k, ref, S):
        kept[(name, j, k)] = pad(ref)
        return kept[(name, j, k)]

    _, _, (da0, _), _ = eq.backward_chain(cats, pad(da3), da3, take)
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())
    errs = {"a3": rel(a3, a3r.detach()), "d(a0)": rel(da0, a0.grad)}
    gslot = lambda j, k: kept[("g5" if k == 5 else "g", j, k)]
    pairs = eq.conv_pairs(s0, cats, gslot, kept[("gpre", 0, 0)], pad(da3))
    assert len(pairs) == 2 + 15 * nb
    for key, a, gk in pairs:
        dw, _, db, _ = eq.wgrad(a, inner(gk))
        errs[f"{key}/W"], errs[f"{key}/b"] = rel(dw, p64[f"{key}/W"].grad), rel(db, p64[f"{key}/b"].grad)
    assert len(errs) == 2 + 2 * (2 + 15 * nb) and all(k in errs for k in params if k.startswith(TRUNK))
    worst = max(errs, key=errs.get)
    print(f"  reference recursion vs oracle autograd: worst {worst} {errs[worst]:.2e}")
    assert errs[worst] <= 1e-12, (worst, errs[worst])


# ---- the checker has teeth ----------------------------------------------------------------------------------------------
def _zero_k_step(w):       # conv3's output channels 0..15: one 16-channel K-step of its data gradient
    w[0:16] = 0
    return w


def _zero_tap(w):
    w[:, :, 0, 0] = 0
    return w


def _conv5_no_high(dw):
    dw[:, 128:192] = 0
    return dw


def _swap_halves(dw):
    return torch.cat([dw[32:64], dw[0:32]], 0)


@pytest.mark.gpu
def test_train_trunk_checker_rejects_wrong_references():
    """Every comparison above fails when fed a deliberately wrong reference; printed: the worst error / bound."""
    step = TrainStep(2, 32, 3, 9, 9, True)
    snap = step.run()
    ok = Report("self-test (right reference)")
    step.check(snap, ok)
    ok.finish()
    lay = step.lay
    tiles = (lay.P + 127) // 128
    assert tiles >= 3
    pos = torch.arange(lay.G0, lay.G0 + lay.P, device="cuda").view(lay.n, lay.Hp, lay.Wp)[:, 1:-1, 1:-1] - lay.G0
    middle = np.array_split(np.arange(tiles), 3)[1]
    drop_split = ((pos // 128 < int(middle[0])) | (pos // 128 > int(middle[-1]))).to(F64).unsqueeze(1)

    def pixel(name, j, k, ref):   # image 1, top row, last column: next to the border
        if (name, j, k) != ("g", 1, 2):
            return ref
        ref = ref.clone()
        c = int(ref[1, :, 0, -1].abs().argmax())
        ref[1, c, 0, -1] += 4 * ulp_bf16(ref[1, c, 0, -1])
        return ref

    def border(ts):
        ts = [t.clone() for t in ts]
        ts[1][0, lay.G0 + 3, 3] = 1.0    # top border row of image 0
        return ts

    cases = [
        ("conv3 dgrad: one 16-channel K-step dropped (block 1)", dict(dgrad_w={(1, 3): _zero_k_step})),
        ("conv5 dgrad: tap (0, 0) dropped (block 4)", dict(dgrad_w={(4, 5): _zero_tap})),
        ("mask of slot a2 ignored (block 3)", dict(mask_off=(3, 2))),
        ("sigma dropped at the r = 3 block 5", dict(sigma={5: 1.0})),
        ("RRDB skip dX_j+3 dropped at block 3", dict(no_rrdb_skip=(3,))),
        ("g2 of block 1, pixel next to the border + 4 bf16 ulps", dict(g_fix=pixel)),
        ("dW of conv2 (block 0) without the middle position split", dict(wgrad_positions={block_key(0, 2): drop_split})),
        ("dW of conv5 (block 2) without channels 128-191", dict(wgrad_fix={block_key(2, 5): _conv5_no_high})),
        ("nonzero border value in a copy of cat[1]", dict(border_fix=border)),
    ]
    wide = TrainStep(2, 64, 3, 9, 9, False)
    wide_snap = wide.run()
    ok = Report("self-test inter 64 (right reference)")
    wide.check(wide_snap, ok)
    ok.finish()
    cases.append(("dW of conv2 (block 1, inter 64) with output halves swapped",
                  dict(wgrad_fix={block_key(1, 2): _swap_halves}), wide, wide_snap))
    for case in cases:
        what, defect = case[:2]
        st, sn = case[2:] if len(case) > 2 else (step, snap)
        rep = Report("self-test")
        st.check(sn, rep, defect)
        assert rep.fails, f"wrong reference accepted: {what}"
        worst = max((w for (_, kind), (w, _, _) in rep.rows.items() if kind != "exact"), default=0.0)
        bad = sum(w for (_, kind), (w, _, _) in rep.rows.items() if kind == "exact")
        if worst > 1.0:
            print(f"  self-test {what:62s} rejected: worst err/bound {worst:10.1f} ({len(rep.fails)} failing checks)")
        else:
            print(f"  self-test {what:62s} rejected: {bad} value(s) differ from the exact expectation")
