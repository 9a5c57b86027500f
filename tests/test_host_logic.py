"""Host-side logic that needs no GPU: the SerialIterator stand-in's epoch wrap-around."""
import numpy as np


def test_array_iterator_completes_last_batch_from_next_epoch():
    """chainer.iterators.SerialIterator(dataset, batch_size, repeat=True, shuffle=True) (srgan_train.py:159-165):
    every batch has batch_size items; a batch reaching the end of the data is completed from the head of the next
    epoch's freshly drawn order, and ``epoch`` advances with that batch."""
    from deepbedmap_b200.train import ArrayIterator
    n, bs = 10, 4
    arrays = {"X": np.arange(n, dtype=np.float32).reshape(n, 1), "Y": np.arange(n, dtype=np.float32)[:, None] * 2}
    it = ArrayIterator(arrays, bs, shuffle=True, seed=3)
    rng = np.random.RandomState(3)
    order0, order1 = rng.permutation(n), rng.permutation(n)
    seen = []
    epochs = []
    for _ in range(5):
        b = it.next()
        assert b["X"].shape == (bs, 1) and np.array_equal(b["Y"], 2 * b["X"])
        seen += [int(v) for v in b["X"][:, 0]]
        epochs.append(it.epoch)
    assert epochs == [0, 0, 1, 1, 2]
    assert seen == list(order0) + list(order1)
    # unshuffled, batch size dividing the data: the epoch flips exactly at the end, nothing is carried over
    it = ArrayIterator(arrays, 5, shuffle=False)
    a, b, c = it.next(), it.next(), it.next()
    assert list(a["X"][:, 0]) == [0, 1, 2, 3, 4] and list(b["X"][:, 0]) == [5, 6, 7, 8, 9] and it.epoch == 1
    assert list(c["X"][:, 0]) == [0, 1, 2, 3, 4]


def test_s2d_tap_mask_matches_the_embedding():
    """flat.s2d_tap_mask: the taps of the 3x3-over-phases embedding of a 4x4 stride-2 filter that touch a real filter
    element (csrc/umma_conv3x3.cu pack mode 2: filter row 2 (ky - 1) + py + 1 in 0..3) -- 4 per phase, their union for
    channel chunks that span phases."""
    from deepbedmap_b200.flat import s2d_tap_mask
    C = 64
    for ph in range(4):
        py, px = ph >> 1, ph & 1
        want = 0
        for tap in range(9):
            ky, kx = 2 * (tap // 3 - 1) + py + 1, 2 * (tap % 3 - 1) + px + 1
            if 0 <= ky <= 3 and 0 <= kx <= 3:
                want |= 1 << tap
        assert bin(want).count("1") == 4
        assert s2d_tap_mask(ph * C, C, C) == want
        assert s2d_tap_mask(ph * C + 16, 32, C) == want
    assert s2d_tap_mask(0, 128, C) == s2d_tap_mask(0, 64, C) | s2d_tap_mask(64, 64, C)
    assert s2d_tap_mask(0, 4 * C, C) == 0x1FF


def test_trunk_plan_pass_sequence():
    """layout.trunk_plan, the trunk pass plan both table builders bind: 2 + 15 nb passes; pair heads / tails (modes 1, 2)
    only when paired at inter_channels 32; no conv5 writes an fp32 buffer it reads; the RRDB skip (res2) exactly on the
    third dense block of each RRDB; and the nb = 1 paired plan, written out."""
    from deepbedmap_b200.layout import trunk_plan
    for nb in (1, 2, 5):
        for inter in (32, 64):
            for paired in (False, True):
                for convs in ((1, 3), (3,), ()):
                    plan = trunk_plan(nb, inter, 0.1, paired and inter == 32, convs)
                    assert len(plan) == 2 + 15 * nb
                    modes = {p["mode"] for p in plan}
                    assert modes == ({0, 1, 2} if paired and inter == 32 and convs else {0})
                    for p in plan:
                        assert p["out_f32"] is None or p["out_f32"] not in (p["res1"], p["res2"])
                        assert (p["res2"] is not None) == p["image"].endswith("residual_dense_block3/conv_layer5")
    fields = ("image", "bias", "cin", "cout", "in_map", "in_cs0", "act", "up2", "out", "out_cs0", "cout_main", "beta",
              "mode", "out_f32", "res1", "res2")
    want = [("pre_residual_conv_layer", "pre_residual_conv_layer/b", 128, 64, 0, 0, 1, 0, "cat0", 0, 64, 0.0, 0, "a1",
             None, None)]
    cat, ring = ["cat0", "cat1", "cat0", "cat1"], [None, "f32_0", "f32_1", "f32_2"]
    res1 = ["a1", "f32_0", "f32_1"]
    for r in (1, 2, 3):
        pre = f"residual_network/0/residual_dense_block{r}"
        c, m = cat[r - 1], 1 + (r - 1) % 2
        want += [(f"{pre}/pair1", f"{pre}/conv_layer1/b", 64, 64, m, 0, 1, 0, c, 8, 32, 0.0, 1, None, None, None),
                 (f"{pre}/tail2", f"{pre}/conv_layer2/b", 32, 32, m, 8, 1, 0, c, 12, 32, 0.0, 2, None, None, None),
                 (f"{pre}/pair3", f"{pre}/conv_layer3/b", 128, 64, m, 0, 1, 0, c, 16, 32, 0.0, 1, None, None, None),
                 (f"{pre}/tail4", f"{pre}/conv_layer4/b", 32, 32, m, 16, 1, 0, c, 20, 32, 0.0, 2, None, None, None),
                 (f"{pre}/conv_layer5", f"{pre}/conv_layer5/b", 192, 64, m, 0, 0, 0, cat[r], 0, 64, 0.25, 0, ring[r],
                  res1[r - 1], "a1" if r == 3 else None)]
    want.append(("post_residual_conv_layer", "post_residual_conv_layer/b", 64, 64, 2, 0, 0, 1, "u1", 0, 64, 1.0, 0, None,
                 "a1", None))
    assert [tuple(p[f] for f in fields) for p in trunk_plan(1, 32, 0.25, True)] == want
