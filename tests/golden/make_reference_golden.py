#!/usr/bin/env python
"""Generates tests/golden/reference_graph_golden.npz by EXECUTING THE REFERENCE'S OWN hot-path code.

/root/reference/srgan_train.py's classes and functions (DeepbedmapInputBlock, ResidualDenseBlock,
ResInResDenseBlock, GeneratorModel, DiscriminatorModel, the four loss / metric functions and both step functions) are
compiled unmodified from the reference tree and run on tests/tools/minichainer.py, a torch-float64 stand-in for the
Chainer 7 / ssim-chainer calls they make (Chainer itself is not installable here: no network, Python 3.12). So these
vectors pin the reference's GRAPH and step logic -- layer wiring, concat order, residual scaling, the detached
adversarial term, eval-mode BatchNorm in the generator step, the constant real labels, the Chainer parameter paths --
by execution; the primitives under them are the shim's restatement of Chainer's documented semantics (SURVEY App. B),
which is why DESIGN.md still calls conv-level VALUES "pinned to the reference's graph, not to Chainer's kernels".

This script reads /root/reference and therefore only runs in the build container; the .npz it writes is committed and
tests/test_reference_graph.py checks the oracle (CPU) and, through the oracle goldens, the CUDA path against it.

Run from the repo root:  python tests/golden/make_reference_golden.py
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "tools"))
import minichainer as mc  # noqa: E402
from oracle import deepbedmap_oracle as O  # noqa: E402  (seeded weights / inputs only)
import importlib.util  # noqa: E402

_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "make_golden.py"))
MG = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(MG)

REFERENCE = "/root/reference/srgan_train.py"
OUT = os.path.join(HERE, "reference_graph_golden.npz")
NAMES = ["DeepbedmapInputBlock", "ResidualDenseBlock", "ResInResDenseBlock", "GeneratorModel", "DiscriminatorModel",
         "calculate_generator_loss", "psnr", "ssim_loss_func", "calculate_discriminator_loss",
         "train_eval_discriminator", "train_eval_generator"]


def build_generator(ns, nb, params):
    g = ns["GeneratorModel"](num_residual_blocks=nb, residual_scaling=0.1)
    x, w1, w2, w3 = O.synthetic_inputs(1)
    with mc.using_config("enable_backprop", False):
        g.forward(x=x, w1=w1, w2=w2, w3=w3)       # materialises the lazily shaped links (in_channels=None)
    mc.load_state(g, params)
    return g


def build_discriminator(ns, params):
    d = ns["DiscriminatorModel"]()
    with mc.using_config("enable_backprop", False), mc.using_config("train", False):
        d.forward(x=np.zeros((1, 1, 36, 36)))
    mc.load_state(d, {k: v for k, v in params.items()})
    return d


def run_reference_tiler():
    """Executes the reference's whole-Antarctica tile-and-predict cell (deepbedmap.py:681-740) verbatim, with a stand-in
    model whose prediction is 'tile index everywhere' and input grids that only record how they are sliced. Returns, per
    tile, the lowres crop [y0, y1, x0, x1] the cell cut for X (with W1/W2/W3 checked to be its 10x / 2x / 1x images) and
    the canvas window [ys, ye, xs, xe] the cell wrote, plus the NaN count of the finished canvas."""
    import ast
    import dataclasses
    import types
    import typing
    src = open("/root/reference/deepbedmap.py").read()
    tree = ast.parse(src)
    body = []
    for node in tree.body:
        if isinstance(node, ast.ClassDef) and node.name == "Shape":
            body.append(node)
        if isinstance(node, ast.With) and "cudnn_deterministic" in ast.get_source_segment(src, node)[:120]:
            body.append(node)
    assert len(body) == 2, "reference tiler cell not found"

    class Grid:   # records slices instead of holding 9.9 GB of REMA
        def __init__(self, scale):
            self.scale = scale

        def __getitem__(self, idx):
            _, _, ys, xs = idx
            return ("crop", self.scale, ys.start, ys.stop, xs.start, xs.stop)

    class FakeModel:
        xp = types.SimpleNamespace(asarray=lambda a, dtype=None: a)
        crops = []

        def forward(self, x, w1, w2, w3):
            _, sc, y0, y1, x0, x1 = x
            assert sc == 1 and w1[1:] == (10, 10 * y0, 10 * y1, 10 * x0, 10 * x1), (x, w1)
            assert w2[1:] == (2, 2 * y0, 2 * y1, 2 * x0, 2 * x1) and w3[1:] == (1, y0, y1, x0, x1), (w2, w3)
            i = len(self.crops)
            self.crops.append((y0, y1, x0, x1))
            return mc.Variable(np.full((1, 1, 4 * (y1 - y0 - 2), 4 * (x1 - x0 - 2)), float(i)))

    model = FakeModel()
    cupy = types.SimpleNamespace(asnumpy=np.asarray)
    ns = {"chainer": mc.as_module(), "np": np, "cupy": cupy, "dataclasses": dataclasses, "typing": typing,
          "model": model, "X_tile": Grid(1), "W1_tile": Grid(10), "W2_tile": Grid(2), "W3_tile": Grid(1)}
    exec(compile(ast.Module(body=body, type_ignores=[]), "/root/reference/deepbedmap.py", "exec"), ns)
    Y_hat = ns["Y_hat"]
    crops = np.array(model.crops, np.int64)
    windows = np.zeros((len(crops), 4), np.int64)
    for i, (y0, y1, x0, x1) in enumerate(crops):
        blk = Y_hat[0, 4 * y0:4 * y1 + 8, 4 * x0:4 * x1 + 8] == float(i)
        rows, cols = np.where(blk.any(1))[0], np.where(blk.any(0))[0]
        assert blk[rows[0]:rows[-1] + 1, cols[0]:cols[-1] + 1].all()
        windows[i] = (4 * y0 + rows[0], 4 * y0 + rows[-1] + 1, 4 * x0 + cols[0], 4 * x0 + cols[-1] + 1)
    covered = int(sum((w[1] - w[0]) * (w[3] - w[2]) for w in windows))
    assert covered == int(np.isfinite(Y_hat).sum()), "tile windows overlap or Y_hat holds stray values"
    return crops, windows, np.array([Y_hat.shape[1], Y_hat.shape[2], int(np.isnan(Y_hat).sum())], np.int64)


def compute() -> dict:
    ns = mc.load_reference_namespace(REFERENCE, NAMES)
    out = {}
    out["tiler/crops"], out["tiler/windows"], out["tiler/canvas"] = run_reference_tiler()
    print("tiler", out["tiler/crops"].shape, out["tiler/canvas"], flush=True)
    # ---- parameter inventory by execution (chainer.serializers.save_npz keys) ----
    g12 = build_generator(ns, 12, O.init_generator_params(12, seed=0))
    sd = mc.state_dict(g12)
    out["inventory/generator_keys"] = np.array(sorted(sd))
    out["inventory/generator_shapes"] = np.array([",".join(map(str, sd[k].shape)) for k in sorted(sd)])
    out["inventory/generator_count_params"] = np.array(g12.count_params())
    d0 = build_discriminator(ns, O.init_discriminator_params(seed=1))
    sdd = mc.state_dict(d0)
    out["inventory/discriminator_keys"] = np.array(sorted(sdd))
    out["inventory/discriminator_count_params"] = np.array(d0.count_params())
    # ---- generator forward on the oracle golden's cases ----
    for name, nb, n, h, w, regime, scale, bias_std in MG.GENERATOR_CASES:
        params, ins = MG.generator_case(nb, n, h, w, regime, scale, bias_std)
        g = build_generator(ns, nb, params)
        with mc.using_config("enable_backprop", False):
            y = g.forward(x=ins[0], w1=ins[1], w2=ins[2], w3=ins[3]).array
        out[f"{name}/y"] = np.array(y)
        print(name, y.shape, float(np.abs(y).max()), flush=True)
    # ---- discriminator: train-mode BN, then eval-mode BN with the updated running statistics ----
    dparams = O.init_discriminator_params(seed=1, bias_std=0.1, scale=1.0)
    d = build_discriminator(ns, dparams)
    x = np.random.RandomState(0).rand(MG.DISC_BATCH, 1, 36, 36).astype(np.float32)
    mc.global_config.train = True
    out["disc/logits_train"] = np.array(d.forward(x=x).array)
    with mc.using_config("train", False):
        out["disc/logits_eval"] = np.array(d.forward(x=x).array)
    out["disc/avg_mean9"] = np.array(d.batch_norm9.avg_mean)
    out["disc/avg_var1"] = np.array(d.batch_norm1.avg_var)
    # ---- the reference's doctest known answers through its own functions ----
    V = mc.Variable
    out["kat/generator_loss"] = np.array(ns["calculate_generator_loss"](
        y_pred=V(np.ones((2, 1, 12, 12))), y_true=np.full((2, 1, 12, 12), 10.0),
        fake_labels=np.array([[-1.2], [0.5]]), real_labels=np.array([[0.5], [-0.8]]),
        fake_minus_real_target=np.array([[1], [1]]).astype(np.int32),
        real_minus_fake_target=np.array([[0], [0]]).astype(np.int32),
        x_topo=np.full((2, 1, 3, 3), 9.0)).array)                                          # srgan_train.py:859-868
    out["kat/psnr"] = np.array(ns["psnr"](y_pred=np.ones((2, 1, 3, 3)), y_true=np.full((2, 1, 3, 3), 2)))  # :916-920
    out["kat/ssim"] = np.array(ns["ssim_loss_func"](y_pred=V(np.ones((2, 1, 9, 9))),
                                                    y_true=np.full((2, 1, 9, 9), 2.0)).array)          # :944-948
    out["kat/discriminator_loss"] = np.array(ns["calculate_discriminator_loss"](
        real_labels_pred=V(np.array([[1.1], [-0.5]])), fake_labels_pred=V(np.array([[-0.3], [1.0]])),
        real_minus_fake_target=np.array([[1], [1]]), fake_minus_real_target=np.array([[0], [0]])).array)  # :985-991
    # ---- one D-step + G-step through the reference's step functions (same case as the oracle golden) ----
    nb, gparams, dparams, arrays = MG.step_case()
    g = build_generator(ns, nb, gparams)
    d = build_discriminator(ns, dparams)
    d_opt = mc.Adam(alpha=1.6e-4, eps=1e-8).setup(d)
    g_opt = mc.Adam(alpha=1.6e-4, eps=1e-8).setup(g)
    dl, da = ns["train_eval_discriminator"](input_arrays=arrays, g_model=g, d_model=d, d_optimizer=d_opt)
    dgr = dict(d.namedparams())
    for k in MG.STEP_GRAD_KEYS_D:
        out[f"step/dgrad/{k}"] = np.array(dgr["/" + k].grad)
    gl, gp, gs = ns["train_eval_generator"](input_arrays=arrays, g_model=g, d_model=d, g_optimizer=g_opt)
    ggr = dict(g.namedparams())
    for k in MG.STEP_GRAD_KEYS_G:
        out[f"step/ggrad/{k}"] = np.array(ggr["/" + k].grad)
    out["step/scalars"] = np.array([dl, da, gl, gp, gs], np.float64)
    out["step/g_after/pre_residual_conv_layer/b"] = np.array(ggr["/pre_residual_conv_layer/b"].array)
    out["step/d_after/linear_2/W"] = np.array(dgr["/linear_2/W"].array)
    print("step", out["step/scalars"], flush=True)
    return out


def main():
    out = compute()
    files = MG.save_golden(OUT, out)
    print(f"wrote {len(out)} arrays to {files}")


if __name__ == "__main__":
    main()
