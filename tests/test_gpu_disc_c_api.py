"""Model-level C entry points of the discriminator (include/deepbedmap_b200.h, dbm_disc_*): forward, backward and
BatchNormalization state through the handle, bit for bit against DiscriminatorModel (the Python composition of the same
kernels), and a complete training step run by a C program that links the library and never touches the Python shim."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import deepbedmap_oracle as O  # noqa: E402  (test infrastructure)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRECISIONS = {"bf16": 0, "fp32": 1}


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


def _keys():
    from deepbedmap_b200 import layout
    params = list(layout.discriminator_shapes())
    persistents = [f"batch_norm{i}/{s}" for i in range(1, 10) for s in ("avg_mean", "avg_var", "N")]
    return params, persistents


def _arrays(seed=1):
    """Seeded parameters (non-zero biases / betas, gammas around 1) and non-trivial running statistics and counters."""
    a = O.init_discriminator_params(seed=seed, bias_std=0.1, scale=1.0)
    rng = np.random.RandomState(seed + 100)
    for i in range(1, 10):
        c = a[f"batch_norm{i}/avg_mean"].shape[0]
        a[f"batch_norm{i}/avg_mean"] = (0.1 * rng.randn(c)).astype(np.float32)
        a[f"batch_norm{i}/avg_var"] = (1.0 + rng.rand(c)).astype(np.float32)
        a[f"batch_norm{i}/N"] = np.array(i, dtype=np.int64)
    return a


def _class(arrays, precision):
    from deepbedmap_b200 import DiscriminatorModel
    d = DiscriminatorModel(precision=precision)
    params, _ = _keys()
    for k in params:
        d.set_param(k, arrays[k])
    for k, t in d.persistent.items():
        t.copy_(torch.from_numpy(arrays[k]))
    for i in range(1, 10):
        d.bn_N[i] = int(arrays[f"batch_norm{i}/N"])
    return d


class Handle:
    """Thin ctypes driver of a dbm_disc handle on torch's current stream (what a C host does)."""

    def __init__(self, precision, arrays=None):
        from deepbedmap_b200 import _lib
        self.lib = _lib.load()
        self.call = _lib.call
        self.h = ctypes.c_void_p()
        self.call("dbm_disc_create", ctypes.byref(self.h))
        self.call("dbm_disc_set_precision", self.h, PRECISIONS[precision])
        self.total = int(self.lib.dbm_disc_count_params(self.h))
        self.info = []
        for i in range(int(self.lib.dbm_disc_num_arrays(self.h))):
            key, ndim, off = ctypes.c_char_p(), ctypes.c_int(), ctypes.c_long()
            dims = (ctypes.c_int * 4)()
            self.call("dbm_disc_array_info", self.h, i, ctypes.byref(key), ctypes.byref(ndim), dims, ctypes.byref(off))
            self.info.append((key.value.decode(), tuple(dims[:ndim.value]), off.value))
        self.shapes = {k: s for k, s, _ in self.info}
        self._ws = {}
        if arrays is not None:
            for k, _, _ in self.info:
                self.set(k, arrays[k])

    def close(self):
        self.call("dbm_disc_destroy", self.h)

    def set(self, key, value):
        v = np.array(np.asarray(value, np.float32).reshape(self.shapes[key]), order="C")   # N stays 0-d
        dims = (ctypes.c_int * 4)(*v.shape)
        self.call("dbm_disc_set_param", self.h, key.encode(), v.ctypes.data, v.ndim, dims)

    def get(self, key):
        torch.cuda.synchronize()
        out = np.empty(self.shapes[key], np.float32)
        self.call("dbm_disc_get_param", self.h, key.encode(), out.ctypes.data)
        return out

    def workspace(self, n, name=0):
        """A 1024-byte aligned device workspace of dbm_disc_workspace_bytes(n): (pointer, bytes)."""
        nbytes = int(self.lib.dbm_disc_workspace_bytes(self.h, n))
        buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device="cuda")
        self._ws[name] = buf
        return (buf.data_ptr() + 1023) & ~1023, nbytes

    def forward(self, x, ws, groups=1, train=True, save=False):
        x = x.contiguous()
        out = torch.empty(x.shape[0], 1, device="cuda")
        self.call("dbm_disc_forward", self.h, x.data_ptr(), x.shape[0], groups, int(train), int(save), out.data_ptr(),
                  ws[0], ws[1], torch.cuda.current_stream().cuda_stream)
        return out

    def backward(self, dlogit, ws):
        self.call("dbm_disc_backward", self.h, dlogit.contiguous().data_ptr(), ws[0], ws[1],
                  torch.cuda.current_stream().cuda_stream)

    def zero_grads(self):
        self.call("dbm_disc_zero_grads", self.h, torch.cuda.current_stream().cuda_stream)


@pytest.fixture
def deterministic():
    from deepbedmap_b200 import train as T
    T.set_deterministic(True)
    yield
    T.set_deterministic(False)


def _stats_equal(h, d):
    for k, t in d.persistent.items():
        assert np.array_equal(h.get(k), t.cpu().numpy()), k


def test_inventory_matches_the_class():
    from deepbedmap_b200 import DiscriminatorModel
    h = Handle("bf16")
    try:
        params, persistents = _keys()
        assert [k for k, _, _ in h.info] == params + persistents
        assert h.total == 10370761 == DiscriminatorModel().count_params()
        d = DiscriminatorModel()
        for k, shp, off in h.info[:len(params)]:
            assert shp == tuple(d.p[k].shape) and off == d._slices[k][0], k
        assert all(off == -1 for _, _, off in h.info[len(params):])
        # a fresh handle starts from Chainer's defaults: gamma 1, beta 0, avg_mean 0, avg_var 1, N 0
        assert np.all(h.get("batch_norm3/gamma") == 1) and np.all(h.get("batch_norm3/beta") == 0)
        assert np.all(h.get("batch_norm3/avg_var") == 1) and np.all(h.get("batch_norm3/avg_mean") == 0)
        assert h.get("batch_norm3/N") == 0
    finally:
        h.close()


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("n,groups", [(1, 1), (6, 1), (6, 2), (256, 1), (256, 2)])
def test_forward_and_running_statistics_equal_the_class(precision, n, groups):
    """Two train forwards in a row, then an eval forward: logits and all 18 running-statistic arrays bit for bit."""
    arrays = _arrays()
    d = _class(arrays, precision)
    h = Handle(precision, arrays)
    try:
        rng = np.random.RandomState(n + groups)
        ws = h.workspace(n)
        for step in range(2):
            x = torch.as_tensor(rng.rand(n, 1, 36, 36).astype(np.float32)).cuda()
            got = h.forward(x, ws, groups=groups, train=True, save=step == 1)
            ref = d.forward(x, train=True, groups=groups).array
            assert torch.equal(got, ref), (step, (got - ref).abs().max().item())
            _stats_equal(h, d)
        got = h.forward(x, ws, groups=groups, train=False)
        assert torch.equal(got, d.forward(x, train=False, groups=groups).array)
        _stats_equal(h, d)
        for i in range(1, 10):   # kept as loaded
            assert h.get(f"batch_norm{i}/N") == i
    finally:
        h.close()


def _bound_grads(h):
    g = torch.zeros(h.total, device="cuda")
    h.call("dbm_disc_bind_grads", h.h, g.data_ptr())
    return g


def _compare_grads(got, ref, exact):
    if exact:
        if not torch.equal(got, ref):
            from deepbedmap_b200 import layout
            off, bad = 0, []
            for k, s in layout.discriminator_shapes().items():
                m = int(np.prod(s))
                if not torch.equal(got[off:off + m], ref[off:off + m]):
                    bad.append(k)
                off += m
            pytest.fail(f"gradients differ: {bad}")
    else:
        assert rel_l2(got.cpu().numpy(), ref.cpu().numpy()) <= 1e-5


@pytest.mark.parametrize("mode", ["deterministic", "default"])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_backward_equals_the_class(request, precision, mode):
    """Stacked D(real) | D(fake) pass with groups = 2 and backward (n = 2 x 128); then two saved passes in two workspaces
    with their backwards in reverse order (the class's two slots); accumulation across backwards; zero_grads.
    Gradients are bit-identical under set_deterministic(True); in the default mode conv_layer0's weight gradient and the
    bias gradients accumulate with float atomics, so they are compared at relative L2 <= 1e-5 there."""
    if mode == "deterministic":
        request.getfixturevalue("deterministic")
    exact = mode == "deterministic"
    arrays = _arrays(seed=3)
    d = _class(arrays, precision)
    h = Handle(precision, arrays)
    try:
        g = _bound_grads(h)
        rng = np.random.RandomState(7)
        n = 128
        real = torch.as_tensor(rng.rand(n, 1, 36, 36).astype(np.float32)).cuda()
        fake = torch.as_tensor(rng.rand(n, 1, 36, 36).astype(np.float32)).cuda()
        dl = torch.as_tensor(rng.randn(2 * n, 1).astype(np.float32)).cuda()
        stacked = torch.cat([real, fake])
        wa, wb = h.workspace(2 * n, "a"), h.workspace(n, "b")
        # stacked pass
        h.zero_grads()
        lg = h.forward(stacked, wa, groups=2, train=True, save=True)
        h.backward(dl, wa)
        d.cleargrads()
        ref = d.forward(stacked, train=True, save=True, groups=2).array
        d.backward(dl)
        torch.cuda.synchronize()
        assert torch.equal(lg, ref)
        _stats_equal(h, d)
        _compare_grads(g, d.flat_grad, exact)
        # accumulation: a second pass on the same batch without zeroing
        h.forward(stacked, wa, groups=2, train=True, save=True)
        h.backward(dl, wa)
        d.forward(stacked, train=True, save=True, groups=2)
        d.backward(dl)
        torch.cuda.synchronize()
        _compare_grads(g, d.flat_grad, exact)
        # two saved passes in flight (two workspaces), backward in reverse order
        h.zero_grads()
        lr = h.forward(real, wb, train=True, save=True)
        wr = h.workspace(n, "r")
        lf = h.forward(fake, wr, train=True, save=True)
        h.backward(dl[n:], wr)
        h.backward(dl[:n], wb)
        rr = d.forward(real, train=True, save=True).array.clone()
        ctx_r = d._ctx
        rf = d.forward(fake, train=True, save=True).array.clone()
        d.cleargrads()
        d.backward(dl[n:])
        d._ctx = ctx_r
        d.backward(dl[:n])
        torch.cuda.synchronize()
        assert torch.equal(lr, rr) and torch.equal(lf, rf)
        _stats_equal(h, d)
        _compare_grads(g, d.flat_grad, exact)
        h.zero_grads()
        torch.cuda.synchronize()
        assert int(torch.count_nonzero(g)) == 0
    finally:
        h.close()


def test_bound_buffers_follow_weight_updates():
    """Bound to the class's flat / flat_grad: a set_param on the class plus dbm_disc_mark_updated reaches the packed
    tensor-core operands of the next forward; backward accumulates into the class's gradient buffer."""
    arrays = _arrays(seed=5)
    d = _class(arrays, "bf16")
    h = Handle("bf16")
    try:
        h.call("dbm_disc_bind_params", h.h, d.flat.data_ptr())
        h.call("dbm_disc_bind_grads", h.h, d.flat_grad.data_ptr())
        _, persistents = _keys()
        for k in persistents:
            h.set(k, arrays[k])
        x = torch.as_tensor(np.random.RandomState(0).rand(8, 1, 36, 36).astype(np.float32)).cuda()
        ws = h.workspace(8)
        y0 = h.forward(x, ws, train=False).clone()
        assert torch.equal(y0, d.forward(x, train=False).array)
        key = "conv_layer4/W"
        d.set_param(key, arrays[key] * 1.5)
        h.call("dbm_disc_mark_updated", h.h)
        y1 = h.forward(x, ws, train=False)
        assert not torch.equal(y0, y1)
        assert torch.equal(y1, d.forward(x, train=False).array)
        d.cleargrads()
        h.forward(x, ws, train=True, save=True)
        h.backward(torch.ones(8, 1, device="cuda"), ws)
        torch.cuda.synchronize()
        assert float(d.flat_grad.abs().sum()) > 0
    finally:
        h.close()


def test_invalid_calls_are_refused_without_launching():
    from deepbedmap_b200 import _lib
    lib = _lib.load()
    h = Handle("bf16", _arrays())
    try:
        st = torch.cuda.current_stream().cuda_stream
        x = torch.rand(6, 1, 36, 36, device="cuda")
        out = torch.empty(6, 1, device="cuda")
        dl = torch.ones(6, 1, device="cuda")
        ws, nbytes = h.workspace(6)
        v = np.zeros(64, np.float32)

        def refused(rc, text=None):
            assert rc == -1
            msg = lib.dbm_last_error().decode()
            assert msg and (text is None or text in msg), msg

        h.forward(x, (ws, nbytes), train=True, save=True)   # tables built, a pass saved
        torch.cuda.synchronize()
        before = _lib.kernel_launches()
        refused(lib.dbm_disc_set_param(h.h, b"no_such_layer/W", v.ctypes.data, 1, (ctypes.c_int * 4)(64)), "unknown key")
        refused(lib.dbm_disc_set_param(h.h, b"batch_norm1/gamma", v.ctypes.data, 1, (ctypes.c_int * 4)(32)), "shape")
        refused(lib.dbm_disc_set_param(h.h, b"batch_norm1/gamma", v.ctypes.data, 2, (ctypes.c_int * 4)(64, 1)), "shape")
        refused(lib.dbm_disc_get_param(h.h, b"no_such_layer/W", v.ctypes.data), "unknown key")
        refused(lib.dbm_disc_forward(h.h, x.data_ptr(), 6, 4, 1, 0, out.data_ptr(), ws, nbytes, st), "groups")
        refused(lib.dbm_disc_forward(h.h, x.data_ptr(), 6, 1, 0, 1, out.data_ptr(), ws, nbytes, st),
                "backward through eval-mode BatchNormalization is not needed by the reference")
        refused(lib.dbm_disc_forward(h.h, x.data_ptr(), 6, 1, 1, 0, out.data_ptr(), ws, nbytes - 1, st), "workspace")
        refused(lib.dbm_disc_forward(h.h, x.data_ptr(), 6, 1, 1, 0, out.data_ptr(), ws + 256, nbytes, st), "aligned")
        refused(lib.dbm_disc_backward(h.h, dl.data_ptr(), ws, nbytes - 1, st), "workspace")
        refused(lib.dbm_disc_backward(h.h, dl.data_ptr(), ws + 1024, nbytes, st), "no saved pass")
        assert _lib.kernel_launches() == before
        h.backward(dl, (ws, nbytes))                         # the saved pass survived the refused calls
        torch.cuda.synchronize()
        before = _lib.kernel_launches()
        refused(lib.dbm_disc_backward(h.h, dl.data_ptr(), ws, nbytes, st), "no saved pass")   # consumed
        assert _lib.kernel_launches() == before
        h.forward(x, (ws, nbytes), train=True, save=False)
        torch.cuda.synchronize()
        before = _lib.kernel_launches()
        refused(lib.dbm_disc_backward(h.h, dl.data_ptr(), ws, nbytes, st), "no saved pass")   # not saved
        assert _lib.kernel_launches() == before
    finally:
        h.close()


def _python_steps(arrays, precision, real, fake, k):
    """The same k steps through the Python composition: train._discriminator_step_enqueue with Adam."""
    from deepbedmap_b200 import train as T
    d = _class(arrays, precision)
    opt = T.Adam().setup(d)
    metrics = []
    for _ in range(k):
        out = T._discriminator_step_enqueue({"Y": real}, None, d, opt, True, False, fake=fake)
        metrics.append(out.cpu().numpy())
    torch.cuda.synchronize()
    final = {k_: d.get_param(k_) for k_ in d.p}
    final.update({k_: t.cpu().numpy() for k_, t in d.persistent.items()})
    final.update({f"batch_norm{i}/N": np.float32(d.bn_N[i]) for i in range(1, 10)})
    return np.concatenate(metrics), final


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_c_host_runs_the_discriminator_training_step(tmp_path, deterministic, precision):
    """tests/c_api/disc_step_main.cu: k = 3 steps of zero_grads -> forward([real; fake], groups 2, save) -> RaGAN loss
    -> backward -> Adam from a C program; losses, accuracies, parameters, running statistics and counters bit for bit
    against the Python step on the same inputs (deterministic mode)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = str(tmp_path / "disc_step_main")
    lib_dir = os.path.join(ROOT, "deepbedmap_b200")
    subprocess.run([nvcc, "-O1", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-o", exe,
                    os.path.join(ROOT, "tests", "c_api", "disc_step_main.cu"), "-L", lib_dir, "-ldeepbedmap_b200",
                    "-Xlinker", "-rpath", "-Xlinker", lib_dir], check=True)
    k, n = 3, 128
    arrays = _arrays(seed=2)
    params, persistents = _keys()
    order = params + persistents
    rng = np.random.RandomState(11)
    real = rng.rand(n, 1, 36, 36).astype(np.float32)
    fake = rng.rand(n, 1, 36, 36).astype(np.float32)
    np.concatenate([np.asarray(arrays[key], np.float32).reshape(-1) for key in order]).tofile(tmp_path / "arrays.bin")
    real.tofile(tmp_path / "real.bin")
    fake.tofile(tmp_path / "fake.bin")
    out = subprocess.run([exe, str(PRECISIONS[precision]), str(k), str(n), str(tmp_path / "arrays.bin"),
                          str(tmp_path / "real.bin"), str(tmp_path / "fake.bin"), str(tmp_path / "out.bin")],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    print(out.stdout.strip())
    res = np.fromfile(tmp_path / "out.bin", np.float32)
    metrics, pos = res[:2 * k], 2 * k
    ref_metrics, ref = _python_steps(arrays, precision, torch.as_tensor(real).cuda(), torch.as_tensor(fake).cuda(), k)
    print(f"C host, {precision}: (d_loss, d_accu) per step {metrics.tolist()}")
    assert np.array_equal(metrics, ref_metrics), (metrics, ref_metrics)
    for key in order:
        m = int(np.prod(np.shape(ref[key])))
        got = res[pos:pos + m].reshape(np.shape(ref[key]))
        pos += m
        assert np.array_equal(got, ref[key]), key
    assert pos == res.size
    assert not np.array_equal(res[2 * k:2 * k + 576], np.asarray(arrays["conv_layer0/W"]).reshape(-1))   # it trained


def test_fp32_handle_matches_the_oracle():
    """The handle's fp32 first-step logits (groups = 2: one BatchNormalization batch per half) against the fp64 oracle,
    as test_discriminator_matches_oracle requires of the class."""
    arrays = _arrays(seed=2)
    rng = np.random.RandomState(11)
    n = 128
    real = rng.rand(n, 1, 36, 36).astype(np.float32)
    fake = rng.rand(n, 1, 36, 36).astype(np.float32)
    h = Handle("fp32", arrays)
    try:
        got = h.forward(torch.as_tensor(np.concatenate([real, fake])).cuda(), h.workspace(2 * n), groups=2,
                        train=True, save=True).cpu().numpy()
    finally:
        h.close()
    p = O.to_torch(arrays)
    ref = np.concatenate([O.discriminator_forward(p, torch.as_tensor(a, dtype=torch.float64), train=True).numpy()
                          for a in (real, fake)])
    err = rel_l2(got, ref)
    print(f"fp32 handle vs fp64 oracle: rel L2 {err:.2e}")
    assert err < 5e-5
