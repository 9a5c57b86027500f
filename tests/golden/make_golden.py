#!/usr/bin/env python
"""Generates tests/golden/hotpath_golden.npz — frozen input/output vectors of the hot path.

Provenance (read this before trusting the file): the reference's arithmetic lives in Chainer 7 /
CuPy / ssim-chainer, none of which is under /root/reference or installable in this image
(SURVEY.md §8c), so these vectors are NOT outputs of the reference itself.  They are outputs of
the float64 CPU oracle (oracle/deepbedmap_oracle.py), which is pinned to every known answer the
reference's own tests hold (tests/test_oracle_kat.py).  Their job is (1) to freeze the oracle: a
later edit to the oracle that changes any value fails tests/test_golden.py on CPU, and (2) to give
the GPU parity tests a fixed target that does not depend on executing oracle code on the GPU box.
Forward/backward values therefore remain "parity unpinned" by the reference (DESIGN.md §2).

Weights and inputs are NOT stored: they are regenerated from seeds (RandomState, key order of
SURVEY App. C); a sha256 of their bytes is stored so a drift of the generators is detected.

Run from the repo root:  python tests/golden/make_golden.py
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import deepbedmap_oracle as O  # noqa: E402

OUT = os.path.join(HERE, "hotpath_golden.npz")
# No stored file exceeds 1 MB: a golden set named <name>.npz is written as shards <name>.<i>.npz of whole arrays, at
# most SHARD_BYTES of array data each (the float data hardly compresses), and read back merged.
SHARD_BYTES = 900_000


def shard_path(path: str, i: int) -> str:
    return f"{path[:-len('.npz')]}.{i}.npz"


def save_golden(path: str, arrays: dict) -> list:
    shards, size = [{}], 0
    for k, v in arrays.items():
        if v.nbytes > SHARD_BYTES:
            raise ValueError(f"{k}: {v.nbytes} bytes do not fit one shard")
        if shards[-1] and size + v.nbytes > SHARD_BYTES:
            shards.append({})
            size = 0
        shards[-1][k] = v
        size += v.nbytes
    for i, s in enumerate(shards):
        np.savez_compressed(shard_path(path, i), **s)
    i = len(shards)
    while os.path.exists(shard_path(path, i)):   # left over from a larger set
        os.remove(shard_path(path, i))
        i += 1
    return [shard_path(path, i) for i in range(len(shards))]


def load_golden(path: str) -> dict:
    out, i = {}, 0
    while os.path.exists(shard_path(path, i)):
        with np.load(shard_path(path, i)) as z:
            out.update({k: z[k] for k in z.files})
        i += 1
    if not out:
        raise FileNotFoundError(f"no shards of {path}")
    return out

# (name, num_residual_blocks, batch, h, w, regime, HeNormal scale, bias_std)
GENERATOR_CASES = [
    ("gen_nb1_doctest", 1, 2, 11, 11, "unit", 1.0, 0.1),
    ("gen_nb2_ragged", 2, 1, 14, 9, "unit", 1.0, 0.1),
    ("gen_nb12_refscale", 12, 1, 11, 11, "unit", 0.1, 0.0),
    ("gen_nb3_wide", 3, 1, 23, 30, "unit", 0.7, 0.1),
]
DISC_BATCH = 6
STEP_BATCH = 3


def digest(arrays) -> str:
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def generator_case(nb, n, h, w, regime, scale, bias_std):
    params = O.init_generator_params(nb, seed=0, bias_std=bias_std, scale=scale)
    ins = O.synthetic_inputs(n, h, w, regime=regime)
    return params, ins


def step_case():
    """One D-step then one G-step on a batch of 3 with a 1-RRDB generator (srgan_train.py:1286-1308)."""
    nb = 1
    gparams = O.init_generator_params(nb, seed=0, bias_std=0.05, scale=1.0)
    dparams = O.init_discriminator_params(seed=1, bias_std=0.1, scale=1.0)
    rng = np.random.RandomState(42)
    n = STEP_BATCH
    arrays = {"X": rng.rand(n, 1, 11, 11), "W1": rng.rand(n, 1, 110, 110), "W2": rng.rand(n, 2, 22, 22),
              "W3": rng.rand(n, 1, 11, 11), "Y": rng.rand(n, 1, 36, 36)}
    arrays = {k: v.astype(np.float32) for k, v in arrays.items()}
    return nb, gparams, dparams, arrays


STEP_GRAD_KEYS_D = ("conv_layer0/W", "conv_layer1/W", "batch_norm3/gamma", "linear_2/b")
STEP_GRAD_KEYS_G = ("final_conv_layer2/deform_conv/W", "post_upsample_conv_layer_1/W",
                    "residual_network/0/residual_dense_block1/conv_layer2/W", "input_block/conv_on_W2/b")


# ---- full-size continent tiles (the configuration bench.py's headline is quoted on) -------------------
# A 3000 x 3000 px sub-continent (752 x 752 lowres grid) has the reference geometry's three tile shapes
# (deepbedmap.py:705-711): corner 269x269, edge 269x288 / 288x269, interior 288x288. Stored: the fp64
# oracle's prediction of a few tiles at 12 RRDB, sub-sampled [::3, ::3] (580 KB per tile), written to a separate
# file so the small fixtures stay small.
TILE_OUT = os.path.join(HERE, "continent_tiles_golden.npz")
TILE_GRID, TILE_FINAL = (752, 752), (3000, 3000)
TILE_STRIDE = 3
STEM_PHYSICAL_SCALE = {"X": 1e-3, "W1": 5e-4, "W2": 5e-3, "W3": 2e-3}
# (name, tile index in the 3x3 plan, HeNormal scale, bias_std, stem filters scaled to the metre-valued inputs)
TILE_CASES = [
    ("bench_interior", 4, 0.1, 0.0, False),      # bench.py's model: GeneratorModel(seed=0), reference init scale
    ("trainedlike_interior", 4, 0.7, 0.1, True),  # O(1) activations: rounding noise is not hidden by tiny residuals
    ("trainedlike_edge", 1, 0.7, 0.1, True),      # 269 x 288 crop (top edge)
]


def tile_params(scale, bias_std, physical, nb=12):
    params = O.init_generator_params(nb, seed=0, bias_std=bias_std, scale=scale)
    if physical:
        for k, f in STEM_PHYSICAL_SCALE.items():
            params[f"input_block/conv_on_{k}/W"] = params[f"input_block/conv_on_{k}/W"] * np.float32(f)
    return params


def compute_tiles() -> dict:
    out = {}
    grids = O.synthetic_continent(TILE_GRID)
    plan = O.tile_plan(TILE_FINAL)
    out["sha_grids"] = np.array(digest(grids))
    for name, idx, scale, bias_std, physical in TILE_CASES:
        params = tile_params(scale, bias_std, physical)
        ins = O.continent_tile_inputs(*grids, plan[idx])
        y = O.generator_forward_numpy(params, *ins, num_residual_blocks=12, fast_deform=True)
        out[f"{name}/y_sub"] = y[0, 0, ::TILE_STRIDE, ::TILE_STRIDE].astype(np.float32)
        out[f"{name}/stats"] = np.array([y.mean(), y.std(), np.abs(y).max(), np.linalg.norm(y[0, 0, ::TILE_STRIDE,
                                                                                             ::TILE_STRIDE])])
        out[f"{name}/shape"] = np.array(y.shape)
        print(name, y.shape, "mean %.4e std %.4e max %.4e" % (y.mean(), y.std(), np.abs(y).max()), flush=True)
    return out


def compute() -> dict:
    out = {}
    for name, nb, n, h, w, regime, scale, bias_std in GENERATOR_CASES:
        params, ins = generator_case(nb, n, h, w, regime, scale, bias_std)
        out[f"{name}/sha_params"] = np.array(digest(params.values()))
        out[f"{name}/sha_inputs"] = np.array(digest(ins))
        out[f"{name}/y"] = O.generator_forward_numpy(params, *ins, num_residual_blocks=nb)
        out[f"{name}/y_bf16_emulated"] = O.generator_forward_numpy(params, *ins, num_residual_blocks=nb,
                                                                   emulate_bf16=True)
    # discriminator: train-mode BN, then eval-mode BN with the updated running statistics
    dparams = O.init_discriminator_params(seed=1, bias_std=0.1, scale=1.0)
    x = np.random.RandomState(0).rand(DISC_BATCH, 1, 36, 36).astype(np.float32)
    p = O.to_torch(dparams)
    stats = {}
    with torch.no_grad():
        out["disc/logits_train"] = O.discriminator_forward(p, torch.as_tensor(x, dtype=torch.float64), train=True,
                                                           stats_out=stats).numpy()
        p.update(stats)
        out["disc/logits_eval"] = O.discriminator_forward(p, torch.as_tensor(x, dtype=torch.float64),
                                                          train=False).numpy()
    out["disc/avg_mean9"] = stats["batch_norm9/avg_mean"].numpy()
    out["disc/avg_var1"] = stats["batch_norm1/avg_var"].numpy()
    out["disc/sha_params"] = np.array(digest(dparams.values()))
    # one training step
    nb, gparams, dparams, arrays = step_case()
    ta = {k: torch.as_tensor(v, dtype=torch.float64) for k, v in arrays.items()}
    gp, dp = O.to_torch(gparams), O.to_torch(dparams)
    dl, da, dgrads = O.train_eval_discriminator(ta, gp, dp, O.ChainerAdam(1.6e-4), num_residual_blocks=nb,
                                                return_grads=True)
    gl, gpsnr, gssim, ggrads = O.train_eval_generator(ta, gp, dp, O.ChainerAdam(1.6e-4), num_residual_blocks=nb,
                                                      return_grads=True)
    out["step/scalars"] = np.array([dl, da, gl, gpsnr, gssim], np.float64)
    for k in STEP_GRAD_KEYS_D:
        out[f"step/dgrad/{k}"] = dgrads[k].numpy()
    for k in STEP_GRAD_KEYS_G:
        out[f"step/ggrad/{k}"] = ggrads[k].numpy()
    return out


def main():
    if "--tiles" in sys.argv or "--all" in sys.argv:
        tiles = compute_tiles()
        files = save_golden(TILE_OUT, tiles)
        print(f"wrote {len(tiles)} arrays to {files}")
        if "--all" not in sys.argv:
            return
    out = compute()
    files = save_golden(OUT, out)
    print(f"wrote {len(out)} arrays to {files}")


if __name__ == "__main__":
    main()
