"""Frozen golden vectors of the hot path (tests/golden/hotpath_golden.npz, made by
tests/golden/make_golden.py — read its header for provenance: they are float64 oracle outputs,
not Chainer outputs, because the reference cannot run in this image).

CPU part (-m "not gpu"): the oracle must still reproduce every frozen value (an edit to the oracle
that changes the arithmetic fails here), and the seeded weight/input generators must not drift.
GPU part (-m gpu): the CUDA path, called through the C ABI shim, against the frozen values with
the tolerances stated in DESIGN.md §2.
"""
import importlib.util
import os

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
MG = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(MG)
O = MG.O


@pytest.fixture(scope="module")
def golden():
    return MG.load_golden(MG.OUT)


def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


def test_oracle_reproduces_golden(golden):
    fresh = MG.compute()
    assert set(fresh) == set(golden)
    for k, v in golden.items():
        if v.dtype.kind == "U":
            assert str(fresh[k]) == str(v), f"seeded generator drifted: {k}"
        else:
            # float64 torch-CPU: the same build reproduces bit for bit; allow reduction-order noise
            # of another BLAS/oneDNN build
            assert fresh[k].shape == v.shape and rel_l2(fresh[k], v) < 1e-9, k


def test_golden_shapes_follow_the_x4_rule(golden):
    for name, nb, n, h, w, *_ in MG.GENERATOR_CASES:
        assert golden[f"{name}/y"].shape == (n, 1, 4 * (h - 2), 4 * (w - 2))   # test_deepbedmap.py:38-39
    assert golden["disc/logits_train"].shape == (MG.DISC_BATCH, 1)            # srgan_train.py:605-606
    assert np.all(np.isfinite(golden["step/scalars"]))


# ------------------------------------------------------------------------------------------
# GPU parity against the frozen vectors
# ------------------------------------------------------------------------------------------
def _load_gen(nb, params, precision):
    from deepbedmap_b200 import GeneratorModel
    m = GeneratorModel(num_residual_blocks=nb, residual_scaling=0.1, precision=precision)
    for k, v in params.items():
        m.set_param(k, v)
    return m


def _load_disc(params, precision="fp32"):
    from deepbedmap_b200 import DiscriminatorModel
    d = DiscriminatorModel(precision=precision)
    for k in d.p:
        d.set_param(k, params[k])
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("case", MG.GENERATOR_CASES, ids=[c[0] for c in MG.GENERATOR_CASES])
def test_generator_fp32_against_golden(golden, case):
    name, nb, n, h, w, regime, scale, bias_std = case
    params, ins = MG.generator_case(nb, n, h, w, regime, scale, bias_std)
    got = _load_gen(nb, params, "fp32").forward(*ins).numpy()
    assert rel_l2(got, golden[f"{name}/y"]) < (1e-4 if nb == 12 else 2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in MG.GENERATOR_CASES if c[6] <= 0.7], ids=lambda c: c[0])
def test_generator_bf16_against_golden(golden, case):
    name, nb, n, h, w, regime, scale, bias_std = case
    params, ins = MG.generator_case(nb, n, h, w, regime, scale, bias_std)
    got = _load_gen(nb, params, "bf16").forward(*ins).numpy()
    ref = golden[f"{name}/y"]
    assert rel_l2(got, golden[f"{name}/y_bf16_emulated"]) < 8e-3
    assert rel_l2(got, ref) < 2e-2 and np.abs(got - ref).max() < 3e-2 * np.abs(ref).max()


@pytest.mark.gpu
def test_discriminator_against_golden(golden):
    dparams = O.init_discriminator_params(seed=1, bias_std=0.1, scale=1.0)
    d = _load_disc(dparams)
    x = np.random.RandomState(0).rand(MG.DISC_BATCH, 1, 36, 36).astype(np.float32)
    assert rel_l2(d.forward(x, train=True).numpy(), golden["disc/logits_train"]) < 5e-5
    assert rel_l2(d.persistent["batch_norm9/avg_mean"].cpu().numpy(), golden["disc/avg_mean9"]) < 1e-5
    assert rel_l2(d.persistent["batch_norm1/avg_var"].cpu().numpy(), golden["disc/avg_var1"]) < 1e-5
    assert rel_l2(d.forward(x, train=False).numpy(), golden["disc/logits_eval"]) < 5e-5


@pytest.mark.gpu
def test_training_step_against_golden(golden):
    from deepbedmap_b200 import train as T
    nb, gparams, dparams, arrays = MG.step_case()
    g = _load_gen(nb, gparams, "fp32")
    d = _load_disc(dparams)
    g_opt, d_opt = T.Adam(1.6e-4).setup(g), T.Adam(1.6e-4).setup(d)
    dl_ref, da_ref, gl_ref, psnr_ref, ssim_ref = golden["step/scalars"]
    dl, da = T.train_eval_discriminator(arrays, g, d, d_opt)
    assert abs(dl - dl_ref) < 1e-4 * max(1, abs(dl_ref)) and abs(da - da_ref) < 1e-6
    for k in MG.STEP_GRAD_KEYS_D:
        ref = golden[f"step/dgrad/{k}"]
        if not np.any(ref):  # RaGAN: d loss / d linear_2/b is exactly 0 (a common logit shift cancels): absolute check
            assert np.abs(d.g[k].cpu().numpy()).max() < 1e-6, k
            continue
        assert rel_l2(d.g[k].cpu().numpy(), ref) < 2e-3, k
    gl, psnr, ssim = T.train_eval_generator(arrays, g, d, g_opt)
    assert abs(gl - gl_ref) < 1e-4 * max(1, abs(gl_ref))
    assert abs(psnr - psnr_ref) < 1e-3 and abs(ssim - ssim_ref) < 1e-4
    for k in MG.STEP_GRAD_KEYS_G:
        tol = 2e-3 if k.startswith("final_conv_layer2") else 2e-2
        assert rel_l2(g.g[k].cpu().numpy(), golden[f"step/ggrad/{k}"]) < tol, k
