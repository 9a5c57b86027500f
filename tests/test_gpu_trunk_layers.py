"""Layer-by-layer value checks of the persistent tensor-core trunk (csrc/umma_trunk.cu) and of two production kernels
that no other test calls directly, each against a float64 reference of the same operation on the kernel's own inputs.

Model-level parity cannot see a wrong trunk layer: every dense-block conv reaches the output through two residual
scalings (beta = 0.1 each) and bf16 storage noise, so a kernel that drops a whole K chunk or tap of one layer still
passes the end-to-end gates. Here each pass is teacher-forced instead:

  * the stem is skipped -- the trunk's input slab s0 is filled with seeded bf16 values;
  * ``dbm_trunk_umma`` runs on a PREFIX of the pass table (the first L records, always ending after a mode-0 record:
    a pair head must be followed by its tail), once per residual dense block (RDB) and once for the whole table;
  * after each prefix every pass of the block just finished is recomputed in float64 (torch on the GPU) from the
    buffers it read, as they are stored: the bf16 feature slabs, the bf16-rounded filter, the fp32 bias and the fp32
    residual streams. The pass table itself (``TRUNK_LAYER_DTYPE`` records) says which buffer and slabs each pass
    reads and writes, and which filter it uses.

Bounds, element-wise (edge bugs touch few pixels; a relative L2 averages them away). S is the float64 convolution of
|x| with |w| (the magnitude of the sum), ulp_bf16(r) the bf16 spacing at |r|:
  fp32 outputs          |got - ref| <= 1e-5 S + 1e-6 |ref|               and relative L2 <= 1e-5
  bf16 outputs          |got - ref| <= ulp_bf16(ref) + 1e-5 S            and relative L2 <= 4e-3
  split hi + lo outputs |got - ref| <= 2^-16 |ref| + 1e-5 S              and relative L2 <= 1e-5
conv5 (and any residual pass with an fp32 output) is compared on its residual BRANCH, (out - res) / beta, because the
skip connection would hide a conv5 error by 1 / beta^2; the unavoidable fp32 rounding of the kernel's two residual
additions (half an fp32 ulp of each partial sum, divided by the branch's scale) is added to that bound. Every bf16
copy of an fp32 result must be exactly its bf16 rounding (split path: exactly its hi / lo split).

The checker has teeth: the self-tests feed the same comparison the reference of a deliberately wrong layer (a dropped
16-channel K chunk, a dropped tap, one unit-edge pixel moved by 4 bf16 ulps) and require it to fail.

Run with -s to see, per layer kind and shape, the worst element error divided by its bound and the relative L2.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import deepbedmap_oracle as O  # noqa: E402  (test infrastructure)

F64 = torch.float64
SLOPE = float(np.float32(0.2))       # kLreluSlope
TOL_REL = {"f32": 1e-5, "bf16": 4e-3, "split": 1e-5}


# ---- element-wise comparison ----------------------------------------------------------------------------------------
def ulp(x, mant_bits):
    """Spacing of a floating-point format with ``mant_bits`` stored mantissa bits at |x| (exact, via frexp)."""
    _, e = torch.frexp(x.abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(x), e - 1 - mant_bits)


def ulp_bf16(x):
    return ulp(x, 7)


def ulp_f32(x):
    return ulp(x, 23)


def bound_of(kind, ref, S):
    if kind == "f32":
        return 1e-5 * S + 1e-6 * ref.abs()
    if kind == "bf16":
        return ulp_bf16(ref) + 1e-5 * S
    if kind == "split":
        return 2.0 ** -16 * ref.abs() + 1e-5 * S
    raise ValueError(kind)


def compare(got, ref, bound):
    """(worst |got - ref| / bound, where, relative L2). NaN / inf in ``got`` count as an infinite error."""
    got, ref = got.to(F64), ref.to(F64)
    diff = got - ref
    ratio = torch.nan_to_num(diff.abs() / bound, nan=float("inf"), posinf=float("inf"))
    k = int(ratio.argmax())
    where = tuple(int(i) for i in np.unravel_index(k, tuple(ratio.shape)))
    rel = float(torch.nan_to_num(diff, nan=float("inf")).norm() / ref.norm().clamp_min(1e-300))
    return float(ratio.reshape(-1)[k]), where, rel


class Report:
    """Per (layer kind, output kind): the worst element error / bound and the worst relative L2 over all passes."""

    def __init__(self, tag):
        self.tag, self.rows, self.fails = tag, {}, []

    def add(self, label, kind, got, ref, bound):
        worst, where, rel = compare(got, ref, bound)
        ok = worst <= 1.0 and rel <= TOL_REL[kind]
        if not ok:
            self.fails.append(f"{label} [{kind}]: worst err/bound {worst:.3g} at {where}, rel L2 {rel:.3g} "
                              f"(limit {TOL_REL[kind]:g})")
        w0, r0, n0 = self.rows.get((label, kind), (0.0, 0.0, 0))
        self.rows[(label, kind)] = (max(w0, worst), max(r0, rel), n0 + 1)

    def exact(self, label, got, want):
        bad = int((got.view(torch.int16) != want.view(torch.int16)).sum())
        if bad:
            self.fails.append(f"{label}: {bad} of {got.numel()} values differ from the exact rounding")
        b0, _, n0 = self.rows.get((label, "exact"), (0, 0.0, 0))
        self.rows[(label, "exact")] = (b0 + bad, 0.0, n0 + 1)

    def finish(self):
        for (label, kind), (worst, rel, n) in sorted(self.rows.items()):
            if kind == "exact":
                print(f"  {self.tag} {label:34s} {n:3d} checks  bit-exact: {'yes' if worst == 0 else f'NO ({worst} differ)'}")
            else:
                print(f"  {self.tag} {label:34s} {n:3d} passes  [{kind:5s}] worst err/bound {worst:.3f}  rel L2 {rel:.2e}")
        for f in self.fails:
            print(f"  {self.tag} FAIL {f}")
        assert not self.fails, self.fails[:5]


# ---- layouts ----------------------------------------------------------------------------------------------------------
def slab8_nchw(t):
    """slab8 [N][C/8][H][W][8] -> NCHW."""
    n, cs, h, w, _ = t.shape
    return t.permute(0, 1, 4, 2, 3).reshape(n, cs * 8, h, w)


def slab8f_nchw(t):
    """The trunk's fp32 side buffers ("slab8f", allocated as (N, 16, H, W, 4)): fp32 [N][8][H][W][8] -> NCHW."""
    n, _, h, w, _ = t.shape
    return slab8_nchw(t.view(n, 8, h, w, 8))


def split_nchw(t):
    """Split-bf16 slab8 buffer, per 16 channels [hi a | hi b | lo a | lo b] slabs -> (hi, lo), each NCHW."""
    n, cs2, h, w, _ = t.shape
    q = t.view(n, cs2 // 4, 4, h, w, 8)
    hi = q[:, :, 0:2].reshape(n, cs2 // 2, h, w, 8)
    lo = q[:, :, 2:4].reshape(n, cs2 // 2, h, w, 8)
    return slab8_nchw(hi), slab8_nchw(lo)


def split_of(v):
    """The kernel's split of fp32 values: hi = bf16(v), lo = bf16(v - hi)."""
    hi = v.bfloat16()
    return hi, (v - hi.float()).bfloat16()


def lrelu(v):
    return torch.where(v >= 0, v, SLOPE * v)


# ---- the trunk, teacher-forced pass by pass ---------------------------------------------------------------------------
def make_model(nb, precision, inter_channels=32, seed=0):
    from deepbedmap_b200 import GeneratorModel
    params = O.init_generator_params(nb, seed=seed, bias_std=0.1, scale=0.7, inter_channels=inter_channels)
    m = GeneratorModel(num_residual_blocks=nb, residual_scaling=0.1, precision=precision, inter_channels=inter_channels)
    for k, v in params.items():
        m.set_param(k, v)
    m.local_trunk = False
    return m


def conv_key(packed_name):
    """Packed-image name of a trunk pass -> the parameter prefix of the conv whose output the pass writes
    (a pair head "pair{k}" writes conv_k, a tail "tail{k}" completes conv_k)."""
    base = packed_name.split("@")[0]
    head, _, last = base.rpartition("/")
    for p in ("pair", "tail"):
        if last.startswith(p):
            return f"{head}/conv_layer{last[len(p):]}"
    return base


class TrunkRun:
    """One trunk workspace with seeded input, run on prefixes of its own pass table."""

    def __init__(self, m, n, H, W, split=False, seed=7):
        from deepbedmap_b200 import ops
        from deepbedmap_b200.model import TRUNK_LAYER_DTYPE
        self.ops, self.m, self.n, self.H, self.W, self.split = ops, m, n, H, W, split
        if split:
            ws = m._split_workspace(n, H, W, m._pack(m.PACK_SPLIT))
            self.table, self.count, self.flags = ws["tables"][0], ws["counts"][0], ws["flags"][0]
            self.fn, self.ccs = "dbm_trunk_umma_split", ws["cat"][0].shape[1] // 2
        else:
            ws = m._trunk_workspace(n, H, W)
            self.table, self.count, self.flags = ws["table"], len(ws["layers"]), ws["flags"]
            self.fn, self.ccs = "dbm_trunk_umma", ws["cat"][0].shape[1]
        self.ws = ws
        self.recs = np.frombuffer(self.table.cpu().numpy().tobytes(), dtype=TRUNK_LAYER_DTYPE)
        assert len(self.recs) == self.count
        names = {v[0].data_ptr(): k for k, v in m._packed.items()
                 if isinstance(v, tuple) and isinstance(v[0], torch.Tensor)}
        self.keys = [conv_key(names[int(r["wpacked"])]) for r in self.recs]
        self.bufs = {ws["s0"].data_ptr(): "s0", ws["cat"][0].data_ptr(): "cat0", ws["cat"][1].data_ptr(): "cat1",
                     ws["a1_f32"].data_ptr(): "a1", ws["u1"].data_ptr(): "u1"}
        for i, t in enumerate(ws["f32"]):
            self.bufs[t.data_ptr()] = f"f32_{i}"
        self.tensors = {"s0": ws["s0"], "cat0": ws["cat"][0], "cat1": ws["cat"][1], "a1": ws["a1_f32"], "u1": ws["u1"],
                        **{f"f32_{i}": t for i, t in enumerate(ws["f32"])}}
        # the trunk's input: seeded N(0, 1) values, as the stem would leave them (bf16, or hi + lo)
        g = torch.Generator(device="cuda").manual_seed(seed)
        x = torch.randn(n, 128, H, W, generator=g, device="cuda")
        if split:
            hi, lo = split_of(x)
            s0 = ws["s0"].view(n, 8, 4, H, W, 8)
            s0[:, :, 0:2] = hi.view(n, 8, 2, 8, H, W).permute(0, 1, 2, 4, 5, 3)
            s0[:, :, 2:4] = lo.view(n, 8, 2, 8, H, W).permute(0, 1, 2, 4, 5, 3)
            assert all(torch.equal(a, b) for a, b in zip(split_nchw(ws["s0"]), (hi, lo)))
        else:
            ws["s0"].copy_(x.bfloat16().view(n, 16, 8, H, W).permute(0, 1, 3, 4, 2))
            assert torch.equal(slab8_nchw(ws["s0"]), x.bfloat16())

    def prefix_ends(self):
        """Last record of every RDB (its conv_layer5) and of the whole table: mode-0 records only."""
        ends = [i for i, k in enumerate(self.keys) if k.endswith("conv_layer5")] + [self.count - 1]
        assert all(int(self.recs[e]["mode"]) == 0 for e in ends)
        return ends

    def run(self, num_layers):
        """Launch the first ``num_layers`` passes; copies of every buffer afterwards."""
        ws, o = self.ws, self.ops
        o.call(self.fn, self.table.data_ptr(), num_layers, self.n, self.H, self.W, ws["s0"].data_ptr(), 16,
               ws["cat"][0].data_ptr(), ws["cat"][1].data_ptr(), self.ccs, self.flags.data_ptr(), o.stream())
        torch.cuda.synchronize()
        return {k: t.clone() for k, t in self.tensors.items()}

    # -- decoding of a snapshot --
    def act_in(self, snap, name):
        """Activation buffer -> float64 NCHW operands: [x] (bf16) or [x_hi, x_lo] (split)."""
        if self.split:
            return [t.to(F64) for t in split_nchw(snap[name])]
        return [slab8_nchw(snap[name]).to(F64)]

    def act_out(self, snap, name):
        """Activation buffer -> (value as stored, float64 NCHW; raw bf16 planes for exactness checks)."""
        if self.split:
            hi, lo = split_nchw(snap[name])
            return hi.to(F64) + lo.to(F64), (hi, lo)
        v = slab8_nchw(snap[name])
        return v.to(F64), (v,)

    def reference(self, xs, w, b):
        """float64 conv (padding 1) + bias of the operands the kernel contracts, and S = conv(|x|, |w|).
        bf16: x . bf16(w); split: x_hi w_hi + x_lo w_hi + x_hi w_lo (the x_lo w_lo term is not computed)."""
        cin = w.shape[1]
        wh = w.bfloat16()
        if self.split:
            wl = (w - wh.float()).bfloat16()
            xh, xl = xs[0][:, :cin], xs[1][:, :cin]
            x = torch.cat([xh, xl, xh], 1)
            wt = torch.cat([wh, wh, wl], 1).to(F64)
        else:
            x, wt = xs[0][:, :cin], wh.to(F64)
        y = F.conv2d(x, wt, padding=1) + b.to(F64).view(1, -1, 1, 1)
        S = F.conv2d(x.abs(), wt.abs(), padding=1)
        return y, S

    def check_pass(self, snap, i, rep, label=None, wfix=None, reffix=None):
        """Recompute pass i of the table from ``snap`` and add its outputs to ``rep``. ``wfix`` / ``reffix`` build a
        deliberately wrong reference (checker self-test)."""
        r, key = self.recs[i], self.keys[i]
        P = self.m.p
        w, b = P[f"{key}/W"].float(), P[f"{key}/b"]
        if wfix is not None:
            w = wfix(w.clone())
        cout = w.shape[0]
        mode = int(r["mode"])
        if label is None:
            label = key.rsplit("/", 1)[-1] + {0: "", 1: " (pair head)", 2: " (pair tail)"}[mode]
        xs = self.act_in(snap, ("s0", "cat0", "cat1")[int(r["in_map"])])
        conv, S = self.reference(xs, w, b)
        if reffix is not None:
            conv = reffix(conv, S)
        act_kind = "split" if self.split else "bf16"
        name = lambda f: self.bufs[int(r[f])] if int(r[f]) else None
        out, out32, res1, res2 = name("out_bf16"), name("out_f32"), name("res1"), name("res2")
        c0 = int(r["out_cs0"]) * 8
        if res1 is None:
            ref = lrelu(conv) if int(r["act"]) else conv
            if out32 is not None:
                got32 = slab8f_nchw(snap[out32])
                rep.add(label + " fp32", "f32", got32, ref, bound_of("f32", ref, S))
                self._check_copy(snap, out, c0, got32, rep, label)
            else:
                got, _ = self.act_out(snap, out)
                got = got[:, c0:c0 + cout]
                rep.add(label, act_kind, got, ref, bound_of(act_kind, ref, S))
            return
        assert not int(r["act"])
        beta = float(r["beta"])
        r1 = slab8f_nchw(snap[res1]).to(F64)
        inner = r1 + beta * conv
        if res2 is not None:
            outv, scale = slab8f_nchw(snap[res2]).to(F64) + beta * inner, beta * beta
            slack = (0.5 * ulp_f32(outv) + beta * 0.5 * ulp_f32(inner)) / scale
        else:
            outv, scale = inner, beta
            slack = 0.5 * ulp_f32(outv) / scale
        if int(r["up2"]):
            # post-residual conv: bf16 (or hi + lo) result, nearest x2 replication fused into the store
            got, raw = self.act_out(snap, out)
            for t in raw:
                q = t[:, c0:c0 + cout]
                for dy, dx in ((0, 1), (1, 0), (1, 1)):
                    rep.exact(label + " x2 replicas", q[:, :, dy::2, dx::2], q[:, :, 0::2, 0::2])
            got = got[:, c0:c0 + cout, 0::2, 0::2]
            rep.add(label, act_kind, got, outv, bound_of(act_kind, outv, S))
            return
        # fp32 result compared on its residual branch: (out - res) / beta (exact res) against conv
        got32 = slab8f_nchw(snap[out32])
        branch = conv + (got32.to(F64) - outv) / scale
        rep.add(label + " fp32 branch", "f32", branch, conv, bound_of("f32", conv, S) + slack)
        self._check_copy(snap, out, c0, got32, rep, label)

    def _check_copy(self, snap, out, c0, got32, rep, label):
        """The bf16 (split: hi / lo) copy the pass stores beside its fp32 result is exactly its rounding."""
        _, raw = self.act_out(snap, out)
        want = split_of(got32) if self.split else (got32.bfloat16(),)
        for t, w_ in zip(raw, want):
            rep.exact(label + " bf16 copy", t[:, c0:c0 + got32.shape[1]], w_)

    def check_all(self, rep):
        """Every pass of the table, one prefix run per RDB plus the whole table."""
        start = 0
        for e in self.prefix_ends():
            snap = self.run(e + 1)
            for i in range(start, e + 1):
                self.check_pass(snap, i, rep)
            start = e + 1
        assert start == self.count


def pairing_limit_exceeded(W):
    return (W + 15) // 16 + 2 > 128


TRUNK_SHAPES = [  # n, H, W: around the 32-row x 16-column work unit and the 148 resident CTAs
    (1, 9, 9),        # narrower than one unit
    (2, 32, 16),      # exact multiples of the unit
    (2, 33, 17),      # one extra row and column of units
    (3, 40, 37),
    (2, 200, 200),    # more units per pass than CTAs
    (4, 286, 286),    # the continent benchmark's batch of 4 interior tiles: 648 units per pass
    (4, 267, 286),    # ... of edge tiles
    (1, 12, 2050),    # wider than the pairing limit: the paired plan falls back to unpaired passes
]


@pytest.mark.parametrize("paired", [True, False], ids=["paired", "unpaired"])
@pytest.mark.parametrize("n,H,W", TRUNK_SHAPES, ids=lambda v: str(v))
def test_trunk_umma_every_pass_matches_fp64(paired, n, H, W):
    """dbm_trunk_umma, nb = 2 (every layer kind: pre-residual, pair heads / tails or plain conv1-4, conv5 with one and
    with two residual streams, post-residual with the fused x2 upsample), each pass against float64 on its inputs."""
    m = make_model(2, "bf16")
    m.paired_trunk = paired
    assert m.paired_convs == (1, 3)   # the production plan
    run = TrunkRun(m, n, H, W)
    modes = set(int(r["mode"]) for r in run.recs)
    assert modes == ({0, 1, 2} if paired and not pairing_limit_exceeded(W) else {0})
    # the slab8f decoding of the fp32 side buffers, once: after the pre-residual pass alone, the bf16 slot a0 is the
    # bf16 rounding of a1_f32 bit for bit
    snap = run.run(1)
    assert torch.equal(slab8_nchw(snap["cat0"])[:, :64], slab8f_nchw(snap["a1"]).bfloat16())
    rep = Report(f"bf16 {'paired' if paired else 'unpaired'} {n}x{H}x{W}")
    run.check_all(rep)
    rep.finish()


@pytest.mark.parametrize("nb,inter,paired,n,H,W", [(12, 32, True, 2, 33, 17), (2, 64, False, 2, 40, 37)],
                         ids=["nb12-paired", "inter64"])
def test_trunk_umma_whole_table_and_wide_blocks(nb, inter, paired, n, H, W):
    """The full 12-RRDB table (182 passes: the flag arrays and the layer-info tables at their production length), and
    the 320-channel dense block of inter_channels = 64 (always unpaired: 64-channel conv1-4 outputs)."""
    m = make_model(nb, "bf16", inter_channels=inter)
    m.paired_trunk = paired
    run = TrunkRun(m, n, H, W)
    assert run.count == 2 + 15 * nb   # pre, 3 nb x (four conv1-4 passes, paired or not, + conv5), post
    rep = Report(f"bf16 nb={nb} inter={inter} {n}x{H}x{W}")
    run.check_all(rep)
    rep.finish()


def test_trunk_checker_rejects_wrong_layers():
    """The comparison above has teeth: fed the reference of a deliberately wrong layer it fails. These are bugs the
    model-level tests cannot see: after two residual scalings they change the generator's output by less than its
    bf16 noise."""
    m = make_model(2, "bf16")
    run = TrunkRun(m, 2, 33, 17)
    i3 = run.keys.index("residual_network/0/residual_dense_block1/conv_layer3")
    i5 = run.keys.index("residual_network/0/residual_dense_block1/conv_layer5")
    assert int(run.recs[i3]["mode"]) == 1
    snap = run.run(i5 + 1)
    ok = Report("self-test (right reference)")
    run.check_pass(snap, i3, ok)
    run.check_pass(snap, i5, ok)
    ok.finish()

    def drop_chunk(w):   # input channels 96..111: one 16-channel K chunk (the first half of a2)
        w[:, 96:112] = 0
        return w

    def drop_tap(w):     # tap (0, 0)
        w[:, :, 0, 0] = 0
        return w

    def edge_pixel(conv, S):   # x = 15 (the last column of the first unit), row 5, image 1, the largest value
        ch = int(conv[1, :, 5, 15].argmax())
        assert conv[1, ch, 5, 15] > 0     # past the LeakyReLU unscaled
        conv = conv.clone()
        conv[1, ch, 5, 15] += 4 * ulp_bf16(conv[1, ch, 5, 15])
        return conv

    cases = [("conv3: K chunk 96-111 dropped", i3, drop_chunk, None), ("conv3: tap (0,0) dropped", i3, drop_tap, None),
             ("conv3: pixel (5, 15) + 4 bf16 ulps", i3, None, edge_pixel),
             ("conv5: K chunk 96-111 dropped", i5, drop_chunk, None), ("conv5: tap (0,0) dropped", i5, drop_tap, None)]
    for what, i, wfix, reffix in cases:
        rep = Report("self-test")
        run.check_pass(snap, i, rep, label=what, wfix=wfix, reffix=reffix)
        assert rep.fails, f"wrong reference accepted: {what}"
        for (label, kind), (worst, rel, _) in rep.rows.items():
            if kind == "exact":   # conv5's bf16 copy of its own (correct) fp32 result
                continue
            print(f"  self-test {label:40s} [{kind:5s}] worst err/bound {worst:9.3f}  rel L2 {rel:.2e} "
                  f"(limit {TOL_REL[kind]:g}): rejected")


# ---- the split-bf16 trunk (precision="bf16x3") -------------------------------------------------------------------------
@pytest.mark.parametrize("n,H,W", [(1, 9, 9), (2, 33, 17), (2, 200, 200), (4, 286, 286)], ids=lambda v: str(v))
def test_trunk_umma_split_every_pass_matches_fp64(n, H, W):
    """dbm_trunk_umma_split, nb = 2: activations as hi + lo bf16 slabs, three MMAs per K chunk; the reference is
    x_hi w_hi + x_lo w_hi + x_hi w_lo in float64, exactly the kernel's stated arithmetic."""
    m = make_model(2, "bf16x3")
    run = TrunkRun(m, n, H, W, split=True)
    assert set(int(r["mode"]) for r in run.recs) == {0, 1, 2}
    snap = run.run(1)
    hi, lo = split_nchw(snap["cat0"])
    want_hi, want_lo = split_of(slab8f_nchw(snap["a1"]))
    assert torch.equal(hi[:, :64], want_hi) and torch.equal(lo[:, :64], want_lo)
    rep = Report(f"bf16x3 {n}x{H}x{W}")
    run.check_all(rep)
    rep.finish()


# ---- conv_on_W1 on the tensor cores: dbm_stem_w1_s2d + dbm_conv3x3_umma_valid ------------------------------------------
def _stem_w1(n, h, w, seed):
    from deepbedmap_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(seed)
    # REMA-like metre-valued input: a smooth relief plus roughness, 0 .. 4000 m
    yy = torch.linspace(0, 6.0, 10 * h, device="cuda").view(-1, 1)
    xx = torch.linspace(0, 6.0, 10 * w, device="cuda").view(1, -1)
    relief = 2000.0 + 1500.0 * torch.sin(yy) * torch.cos(0.7 * xx)
    w1 = (relief + 400.0 * torch.rand(n, 1, 10 * h, 10 * w, generator=g, device="cuda")).clamp(0.0, 4000.0)
    # HeNormal(0.7) filter scaled by the inverse input range, as a trained model's would be
    filt = torch.randn(32, 1, 30, 30, generator=g, device="cuda") * (0.7 * (2.0 / 900) ** 0.5 * 5e-4)
    bias = torch.randn(32, generator=g, device="cuda") * 0.1
    s2d = ops.empty(n, 40, h, w, 8, dtype=torch.bfloat16)
    packed = ops.empty(9 * 320 * 32, dtype=torch.bfloat16)
    s0 = torch.full((n, 16, h - 2, w - 2, 8), 7.0, dtype=torch.bfloat16, device="cuda")
    st = ops.stream()
    ops.call("dbm_pack_stem_w1", filt.data_ptr(), packed.data_ptr(), st)
    ops.call("dbm_stem_w1_s2d", w1.data_ptr(), s2d.data_ptr(), n, h, w, st)
    ops.call("dbm_conv3x3_umma_valid", s2d.data_ptr(), 40, 320, packed.data_ptr(), bias.data_ptr(), n, h, w,
             s0.data_ptr(), 16, 4, st)
    torch.cuda.synchronize()
    return w1, filt, bias, s0


@pytest.mark.parametrize("n,h,w", [(2, 11, 11), (1, 23, 37), (3, 36, 19), (1, 290, 290)], ids=lambda v: str(v))
def test_stem_w1_tensor_core_matches_fp64(n, h, w):
    """conv_on_W1 (k30 s10, 99 % of the stem's FLOPs) as a split-bf16 tcgen05 GEMM over the 10x10 space-to-depth:
    channels 32-63 of s0 against float64 conv2d(W1, W, b, stride=10) on metre-scale input. Bound: one bf16 rounding
    of the output + 2^-16 S. Losing the x_lo term costs about 2^-9 S, which the bound rejects (shown below with
    the reference of that arithmetic)."""
    w1, filt, bias, s0 = _stem_w1(n, h, w, seed=h * 1000 + w)
    got = slab8_nchw(s0)
    x, f = w1.to(F64), filt.to(F64)
    ref = F.conv2d(x, f, bias.to(F64), stride=10)
    S = F.conv2d(x.abs(), f.abs(), stride=10)
    assert got.shape[1:] == (128, h - 2, w - 2)
    assert torch.all(got[:, :32] == 7.0) and torch.all(got[:, 64:] == 7.0)   # the other stem channels untouched
    worst, where, rel = compare(got[:, 32:64], ref, ulp_bf16(ref) + 2.0 ** -16 * S)
    print(f"  stem W1 {n}x{h}x{w}: worst err/bound {worst:.3f} at {where}, rel L2 {rel:.2e}, "
          f"median S/|ref| {float((S / ref.abs().clamp_min(1e-30)).median()):.1f}")
    assert worst <= 1.0 and rel <= 4e-3
    # self-test: the plain bf16 product (x_hi w_hi, no lo terms) is rejected by the same bound
    q = lambda t: t.bfloat16().to(F64)
    wrong = F.conv2d(q(w1), q(filt), bias.to(F64), stride=10)
    worst_w, where_w, _ = compare(got[:, 32:64], wrong, ulp_bf16(ref) + 2.0 ** -16 * S)
    print(f"  stem W1 {n}x{h}x{w} self-test (reference without the lo terms): worst err/bound {worst_w:.3f} at "
          f"{where_w}: rejected")
    assert worst_w > 1.0


# ---- training forward of the first deformable layer: dbm_deform_conv_umma_nchw -----------------------------------------
@pytest.mark.parametrize("n,h,w", [(2, 37, 45), (1, 20, 52), (128, 36, 36)], ids=lambda v: str(v))
def test_deform_conv_fused_forward_matches_fp64(n, h, w):
    """ops.deform_conv_fwd_fused (gather -> tcgen05 -> bias + LeakyReLU, fp32 NCHW output) against the float64
    contraction of bf16(deform_sample_slab8(...)) -- the samples of the same bf16 input with the same blend -- with
    the bf16 filter, plus bias and LReLU. Offsets include samples far outside the image, integer offsets (exact
    corner hits) and samples straddling the border."""
    from deepbedmap_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(n * 100 + h)
    x = torch.randn(n, 64, h, w, generator=g, device="cuda")
    off = torch.randn(n, 18, h, w, generator=g, device="cuda") * 1.5
    off[0, :, 0, 0] = 50.0                      # far outside: every corner clamped, zero weight
    off[0, :9, 1, 1] = -30.0
    off[0, :, 2, 3] = torch.tensor([float(v) for v in (-2, -1, 0, 1, 2, 3, -3, 1, -1) * 2], device="cuda")  # integers
    off[0, :9, 4, 0] = -0.5                     # x straddles the left border
    off[0, 9:, 0, 5] = -0.75                    # y straddles the top border
    off[-1, :9, h - 1, w - 1] = 0.5             # bottom-right corner pixel, half a pixel beyond the right border
    off[-1, 9:, h - 2, 7] = 1.25                # ... beyond the bottom border
    wt = torch.randn(64, 64, 3, 3, generator=g, device="cuda") * 0.1
    b = torch.randn(64, generator=g, device="cuda")
    y, x8 = ops.deform_conv_fwd_fused(x, off, ops.pack_conv3x3(wt, 64, ck=64), b, act=True, keep_slab8=True)
    cols = ops.deform_sample_slab8(x8, off)     # (n, 576, hw): index c * 9 + tap
    torch.cuda.synchronize()
    q = lambda t: t.bfloat16().to(F64)
    wm = q(wt.reshape(64, 576))
    ref = lrelu(torch.einsum("nkp,ok->nop", q(cols), wm) + b.to(F64).view(1, 64, 1)).view(n, 64, h, w)
    S = torch.einsum("nkp,ok->nop", q(cols).abs(), wm.abs()).view(n, 64, h, w)
    worst, where, rel = compare(y, ref, bound_of("f32", ref, S))
    print(f"  deform fused forward {n}x{h}x{w}: worst err/bound {worst:.3f} at {where}, rel L2 {rel:.2e}")
    assert y.shape == (n, 64, h, w)
    assert worst <= 1.0 and rel <= 1e-5
