"""The oracle against vectors produced by EXECUTING THE REFERENCE'S OWN CODE (tests/golden/reference_graph_golden.npz:
srgan_train.py's model classes, loss functions and step functions compiled unmodified from the reference tree and
run on a float64 stand-in for the Chainer calls they make -- tests/golden/make_reference_golden.py,
tests/tools/minichainer.py). What this pins that the restated oracle alone could not: the graph wiring, the step
functions' detach / eval-BatchNorm / constant-label logic and the Chainer parameter paths, by execution of the
reference's lines. The CUDA path is checked against the oracle goldens (tests/test_golden.py), which this file ties
to the reference-executed ones value by value.

CPU only; nothing here reads /root/reference (the vectors are committed).
"""
import importlib.util
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
MG = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(MG)


@pytest.fixture(scope="module")
def ref():
    return MG.load_golden(os.path.join(HERE, "golden", "reference_graph_golden.npz"))


@pytest.fixture(scope="module")
def ora():
    return MG.load_golden(MG.OUT)


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


def test_parameter_paths_are_the_references_own(ref):
    """chainer.serializers.save_npz keys = link paths of the reference's Chain attributes, here obtained by building
    the reference's classes; the product's layout (deepbedmap_b200/layout.py, SURVEY App. C) must be that set."""
    from deepbedmap_b200 import layout
    shapes = layout.generator_shapes(12)
    assert sorted(shapes) == [str(k) for k in ref["inventory/generator_keys"]]
    for k, s in zip(ref["inventory/generator_keys"], ref["inventory/generator_shapes"]):
        assert tuple(int(v) for v in str(s).split(",")) == tuple(shapes[str(k)]), k
    assert int(ref["inventory/generator_count_params"]) == 8907749              # srgan_train.py:446-447
    d_keys = set(layout.discriminator_shapes()) | set(layout.discriminator_persistents())
    d_keys |= {f"batch_norm{i}/N" for i in range(1, 10)}
    assert d_keys == {str(k) for k in ref["inventory/discriminator_keys"]}
    assert int(ref["inventory/discriminator_count_params"]) == 10370761         # srgan_train.py:607-608


def test_reference_doctest_values_through_reference_functions(ref):
    assert abs(float(ref["kat/generator_loss"]) - 4.35108415) < 1e-8            # srgan_train.py:868
    assert abs(float(ref["kat/psnr"]) - 192.65919722494797) < 1e-9              # :920
    assert abs(float(ref["kat/ssim"]) - 0.800004) < 1e-6                        # :948
    assert abs(float(ref["kat/discriminator_loss"]) - 1.56670504) < 1e-8        # :991


def test_oracle_generator_equals_reference_graph(ref, ora):
    for name in ("gen_nb1_doctest", "gen_nb2_ragged", "gen_nb12_refscale", "gen_nb3_wide"):
        assert ref[f"{name}/y"].shape == ora[f"{name}/y"].shape
        assert rel_l2(ora[f"{name}/y"], ref[f"{name}/y"]) < 1e-10, name


def test_oracle_discriminator_equals_reference_graph(ref, ora):
    for k in ("disc/logits_train", "disc/logits_eval", "disc/avg_mean9", "disc/avg_var1"):
        assert rel_l2(ora[k], ref[k]) < 1e-10, k


def test_oracle_training_step_equals_reference_step_functions(ref, ora):
    """train_eval_discriminator then train_eval_generator of the reference (srgan_train.py:1084-1263) on a batch of 3:
    losses / metrics and parameter gradients of both models."""
    assert np.allclose(ora["step/scalars"], ref["step/scalars"], rtol=1e-9, atol=1e-12)
    keys = [k for k in ref if k.startswith("step/dgrad/") or k.startswith("step/ggrad/")]
    assert len(keys) == 8
    for k in keys:
        assert rel_l2(ora[k], ref[k]) < 1e-8, k


def test_tile_geometry_is_the_reference_cells_own(ref):
    """deepbedmap.py:681-740 executed verbatim on recording stand-ins: the lowres crop of every one of the 396 tiles and
    the canvas window it is written to (incl. the 4-px placement offset and the NaN frame) -- the product's and the
    oracle's tile plans must be exactly that."""
    from deepbedmap_b200.tiler import tile_plan
    from oracle import deepbedmap_oracle as O
    crops, windows, canvas = ref["tiler/crops"], ref["tiler/windows"], ref["tiler/canvas"]
    plan = tile_plan()
    assert len(plan) == len(crops) == 396 and tuple(canvas[:2]) == (18000, 22000)
    for t, c, w in zip(plan, crops, windows):
        assert tuple(t[:4]) == tuple(int(v) for v in c) and tuple(t[4:]) == tuple(int(v) for v in w)
    for t, c, w in zip(O.tile_plan(), crops, windows):
        assert tuple(t[:4]) == tuple(int(v) for v in c)
        assert (t[4].start, t[4].stop, t[5].start, t[5].stop) == tuple(int(v) for v in w)
    # the reference leaves the outermost 76 px NaN: 18000*22000 - (18000-152)*(22000-152) pixels
    assert int(canvas[2]) == 18000 * 22000 - (18000 - 152) * (22000 - 152)
    shapes = {(int(c[1] - c[0]), int(c[3] - c[2])) for c in crops}
    assert shapes == {(288, 288), (269, 288), (288, 269), (269, 269)}
