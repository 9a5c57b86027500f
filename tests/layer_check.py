"""Element-wise comparison of a kernel's output with a float64 reference, shared by the layer-by-layer value checks
(test_gpu_trunk_layers.py, test_gpu_train_trunk_layers.py).

Bounds, element-wise (edge bugs touch few pixels; a relative L2 averages them away). S is the float64 contraction of
the operands' magnitudes (the magnitude of the sum), ulp_bf16(r) the bf16 spacing at |r|:
  fp32 outputs          |got - ref| <= 1e-5 S + 1e-6 |ref|               and relative L2 <= 1e-5
  bf16 outputs          |got - ref| <= ulp_bf16(ref) + 1e-5 S            and relative L2 <= 4e-3
  split hi + lo outputs |got - ref| <= 2^-16 |ref| + 1e-5 S              and relative L2 <= 1e-5
"""
import numpy as np
import torch

F64 = torch.float64
TOL_REL = {"f32": 1e-5, "bf16": 4e-3, "split": 1e-5}


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

    def add(self, label, kind, got, ref, bound, rel_limit=None):
        """``rel_limit``: relative-L2 cap when it is not TOL_REL[kind] (results compared on a branch)."""
        worst, where, rel = compare(got, ref, bound)
        limit = TOL_REL[kind] if rel_limit is None else rel_limit
        ok = worst <= 1.0 and rel <= limit
        if not ok:
            self.fails.append(f"{label} [{kind}]: worst err/bound {worst:.3g} at {where}, rel L2 {rel:.3g} "
                              f"(limit {limit:.3g})")
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
