"""Value parity of the configuration the headline benchmark is quoted on (BASELINE.json configs[2]):
full-size continent tiles -- interior 288x288, edge 269x288, corner 269x269 lowres crops (deepbedmap.py:705-711) --
through the 12-RRDB generator on the bf16 tensor-core path in batches of 4 (648 work items per trunk pass, so every
one of the 148 persistent CTAs takes several items of one pass), against

  * the fp64 CPU oracle's prediction of the same tiles, generated offline by tests/golden/make_golden.py --tiles
    (tests/golden/continent_tiles_golden.npz; nothing of oracle/ is timed or shipped here, it is the checker);
  * the exact-arithmetic fp32 CUDA path of the same library (itself <= 1e-4 from the golden).

Stated tolerances: bf16 path relative L2 <= 2e-2 and max-abs <= 3e-2 of the output range vs fp64 (DESIGN.md
"Numerics"); fp32 path relative L2 <= 1e-4. Errors are also printed in METRES for an output calibrated to BEDMAP2's
spread (the synthetic weights are random, so the raw output unit is arbitrary: metres = error / std(output) * 800 m,
800 m being the standard deviation of the synthetic bed-elevation input X; run with -s to see them, the GPU log of
the round is committed under profiles/).
"""
import importlib.util
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import deepbedmap_oracle as O  # noqa: E402  (test infrastructure)

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
MG = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(MG)
GOLD = MG.TILE_OUT
GRID, FINAL, STRIDE = (752, 752), (3000, 3000), 3
STEM_PHYSICAL_SCALE = {"X": 1e-3, "W1": 5e-4, "W2": 5e-3, "W3": 2e-3}
CASES = {  # name -> (tile index, HeNormal scale, bias_std, stem filters scaled to metre-valued inputs)
    "bench_interior": (4, 0.1, 0.0, False),
    "trainedlike_interior": (4, 0.7, 0.1, True),
    "trainedlike_edge": (1, 0.7, 0.1, True),
}
BED_STD_M = 800.0


def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


@pytest.fixture(scope="module")
def grids():
    return O.synthetic_continent(GRID)


@pytest.fixture(scope="module")
def gold():
    return MG.load_golden(GOLD)


def make_model(scale, bias_std, physical, precision, nb=12):
    from deepbedmap_b200 import GeneratorModel
    params = O.init_generator_params(nb, seed=0, bias_std=bias_std, scale=scale)
    if physical:
        for k, f in STEM_PHYSICAL_SCALE.items():
            params[f"input_block/conv_on_{k}/W"] = params[f"input_block/conv_on_{k}/W"] * np.float32(f)
    m = GeneratorModel(num_residual_blocks=nb, residual_scaling=0.1, precision=precision)
    for k, v in params.items():
        m.set_param(k, v)
    return m


@pytest.mark.parametrize("case", list(CASES))
def test_full_size_tile_batch4_matches_oracle_golden(case, grids, gold):
    idx, scale, bias_std, physical = CASES[case]
    plan = O.tile_plan(FINAL)
    crop = O.continent_tile_inputs(*grids, plan[idx])
    h, w = crop[0].shape[2:]
    assert (h, w) == ((288, 288) if idx == 4 else (269, 288))
    # batch of 4 as the tiler forms it: slot 2 is the golden tile, the other slots carry different data
    # (rolled copies) so that any cross-image mix-up in the work-item bookkeeping shows
    batch = [np.concatenate([np.roll(a, s * 7 * (a.shape[2] // h), axis=2) for s in (1, 2, 0, 3)]) for a in crop]
    ref_sub = gold[f"{case}/y_sub"]
    _, std, amax, _ = gold[f"{case}/stats"]
    m16 = make_model(scale, bias_std, physical, "bf16")
    y16 = m16.forward(*batch).array
    assert tuple(y16.shape) == (4, 1, 4 * (h - 2), 4 * (w - 2))
    # the persistent kernel's flag protocol: a tile computed alone (162 items per pass) and inside the batch
    # (648 items per pass, dealt to the same 148 CTAs in a different order) must agree bit for bit
    alone = m16.forward(*crop).array
    assert torch.equal(alone[0], y16[2])
    for _ in range(2):
        assert torch.equal(m16.forward(*batch).array, y16)
    got16 = y16[2, 0].cpu().numpy()
    m32 = make_model(scale, bias_std, physical, "fp32")
    got32 = m32.forward(*crop).array[0, 0].cpu().numpy()
    e32 = rel_l2(got32[::STRIDE, ::STRIDE], ref_sub)
    e16 = rel_l2(got16[::STRIDE, ::STRIDE], ref_sub)
    e16_32 = rel_l2(got16, got32)
    max16 = float(np.abs(got16[::STRIDE, ::STRIDE] - ref_sub).max())
    max32 = float(np.abs(got32[::STRIDE, ::STRIDE] - ref_sub).max())
    max16_32 = float(np.abs(got16 - got32).max())
    to_m = BED_STD_M / std
    print(f"\n[{case}] {h}x{w} crop, 12 RRDB, output std {std:.4e} max {amax:.4e}\n"
          f"   fp32 path vs fp64 golden : rel_l2 {e32:.3e}  max_abs {max32:.3e} = {max32 * to_m:.4f} m\n"
          f"   bf16 path vs fp64 golden : rel_l2 {e16:.3e}  max_abs {max16:.3e} = {max16 * to_m:.3f} m "
          f"(rms {e16 * np.sqrt((ref_sub ** 2).mean()) * to_m:.3f} m)\n"
          f"   bf16 path vs fp32 path   : rel_l2 {e16_32:.3e}  max_abs {max16_32:.3e} = {max16_32 * to_m:.3f} m")
    assert e32 < 1e-4
    assert e16 < 2e-2 and e16_32 < 2e-2
    assert max16 < 3e-2 * amax


def test_predict_continent_bf16_batch4_matches_fp32_path(grids):
    """The tiler as bench.py drives it (bench model: GeneratorModel(seed=0), reference init; batch_tiles=4, all
    three tile shapes, NaN frame, 4-px placement offset) against the exact fp32 path run tile by tile."""
    from deepbedmap_b200 import GeneratorModel, predict_continent
    kw = dict(final_shape=FINAL, ary_shape=(1000, 1000), stride=(1000, 1000), xtrapad=(18, 18))
    m16 = GeneratorModel(num_residual_blocks=12, residual_scaling=0.1, precision="bf16", seed=0)
    m32 = GeneratorModel(num_residual_blocks=12, residual_scaling=0.1, precision="fp32", seed=0)
    y16 = predict_continent(m16, *grids, batch_tiles=4, **kw)
    y32 = predict_continent(m32, *grids, batch_tiles=1, **kw)
    assert y16.shape == y32.shape == (1, 3000, 3000)
    nan16, nan32 = np.isnan(y16), np.isnan(y32)
    assert np.array_equal(nan16, nan32)
    # the reference's NaN frame: the outermost 76 output px are never written (deepbedmap.py:696, 731-736)
    assert nan16[0, :76].all() and nan16[0, :, :76].all() and not nan16[0, 76:-76, 76:-76].any()
    a, b = y16[~nan16], y32[~nan32]
    err, mx, std = rel_l2(a, b), float(np.abs(a - b).max()), float(b.std())
    print(f"\n[sub-continent 3000x3000, 9 tiles] bf16/batch 4 vs fp32/batch 1: rel_l2 {err:.3e} max_abs {mx:.3e} "
          f"(output std {std:.3e}) = {mx / std * BED_STD_M:.3f} m for an 800 m output spread")
    assert err < 2e-2
    # same through the int16 product path (deepbedmap.py:751): identical to astype on the float canvas
    y16i = predict_continent(m16, *grids, batch_tiles=4, out_dtype="int16", **kw)
    with np.errstate(invalid="ignore"):
        assert np.array_equal(y16i, predict_continent(m16, *grids, batch_tiles=4, **kw).astype(np.int16))


def test_persistent_trunk_more_items_than_ctas_equals_per_layer_launches():
    """> 148 work items per pass (2 x 13 x 7 = 182 units of 32 x 16 px): every CTA of the persistent kernel takes more
    than one item of a pass; must equal the per-layer launches bit for bit (same MMAs, same order)."""
    from deepbedmap_b200 import GeneratorModel
    params = O.init_generator_params(1, seed=0, bias_std=0.1, scale=0.7)
    m = GeneratorModel(num_residual_blocks=1, precision="bf16")
    for k, v in params.items():
        m.set_param(k, v)
    m.local_trunk = False
    ins = O.synthetic_inputs(2, 200, 200)
    m.persistent_trunk, m.per_layer_ck16 = False, True
    ref = m.forward(*ins).array.clone()
    m.persistent_trunk, m.paired_trunk = True, False
    for _ in range(3):
        assert torch.equal(m.forward(*ins).array, ref)
    m.paired_trunk = True
    first = m.forward(*ins).array.clone()
    assert torch.equal(m.forward(*ins).array, first)
    assert rel_l2(first.cpu().numpy(), ref.cpu().numpy()) < 8e-3


@pytest.mark.parametrize("case", ["bench_interior", "trainedlike_edge"])
def test_split_bf16_path_matches_oracle_golden(case, grids, gold):
    """precision="bf16x3" (split-bf16 trunk + upsample convs on the tensor cores, stem and deformable layers fp32): the
    full-size tile against the fp64 golden and against the fp32 CUDA path -- fp32-grade: relative L2 <= 1e-4 (stated);
    a tile in a batch of 2 equals the tile alone bit for bit."""
    idx, scale, bias_std, physical = CASES[case]
    plan = O.tile_plan(FINAL)
    crop = O.continent_tile_inputs(*grids, plan[idx])
    h, w = crop[0].shape[2:]
    batch = [np.concatenate([np.roll(a, 5 * (a.shape[2] // h), axis=2), a]) for a in crop]
    ref_sub = gold[f"{case}/y_sub"]
    _, std, amax, _ = gold[f"{case}/stats"]
    m3 = make_model(scale, bias_std, physical, "bf16x3")
    y3 = m3.forward(*batch).array
    assert tuple(y3.shape) == (2, 1, 4 * (h - 2), 4 * (w - 2))
    alone = m3.forward(*crop).array
    assert torch.equal(alone[0], y3[1])
    got3 = y3[1, 0].cpu().numpy()
    e3 = rel_l2(got3[::STRIDE, ::STRIDE], ref_sub)
    max3 = float(np.abs(got3[::STRIDE, ::STRIDE] - ref_sub).max())
    to_m = BED_STD_M / std
    print(f"\n[{case}] bf16x3 path vs fp64 golden: rel_l2 {e3:.3e}  max_abs {max3:.3e} = {max3 * to_m:.4f} m")
    assert e3 < 1e-4
    assert max3 * to_m < 1.0   # sub-metre for an output calibrated to BEDMAP2's 800 m spread
