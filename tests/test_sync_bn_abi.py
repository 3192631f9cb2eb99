"""CPU: argument validation of the split BatchNorm entry points behind SyncBatchNorm (ffb6d_bn_train_stats /
_apply / _bwd_stats / _bwd_apply).  Every rejected call returns before any CUDA work, so no GPU is needed."""
import ctypes as C

from ffb6d_b200 import _lib

ERR = _lib.ERR_INVALID


def _buffers():
    raw = (C.c_double * 256)()
    base = (C.addressof(raw) + 15) & ~15        # 16-byte aligned, as stats must be
    return raw, base


def test_bn_train_stats_validation():
    lib = _lib.lib
    raw, p = _buffers()
    ws = 1 << 20
    assert lib.ffb6d_bn_train_stats(p, 0, 4, 8, p, p, ws, None) == ERR and "bad size" in _lib.last_error()
    assert lib.ffb6d_bn_train_stats(p, 1, 65536, 8, p, p, ws, None) == ERR
    assert lib.ffb6d_bn_train_stats(p, 65536, 1, 8, p, p, ws, None) == ERR
    assert lib.ffb6d_bn_train_stats(p, 1, 4, 1 << 31, p, p, ws, None) == ERR
    assert lib.ffb6d_bn_train_stats(None, 1, 4, 8, p, p, ws, None) == ERR and "null" in _lib.last_error()
    assert lib.ffb6d_bn_train_stats(p, 1, 4, 8, None, p, ws, None) == ERR
    assert lib.ffb6d_bn_train_stats(p, 1, 4, 8, p, None, ws, None) == ERR
    assert lib.ffb6d_bn_train_stats(p, 1, 4, 8, p + 4, p, ws, None) == ERR and "aligned" in _lib.last_error()
    assert lib.ffb6d_bn_train_stats(p, 1, 4, 8, p, p, 0, None) == ERR and "workspace" in _lib.last_error()


def test_bn_train_apply_validation():
    lib = _lib.lib
    raw, p = _buffers()

    def apply(B=2, C_=4, P=8, z=p, sums=p, count=16.0, act=1, stats=p, y=p):
        return lib.ffb6d_bn_train_apply(z, B, C_, P, sums, count, p, p, 1e-5, 0.1, p, p, act, 0.0, stats, y, None)

    assert apply(C_=0) == ERR and "bad size" in _lib.last_error()
    assert apply(P=0) == ERR
    assert apply(z=None) == ERR and "null" in _lib.last_error()
    assert apply(sums=None) == ERR
    assert apply(stats=None) == ERR
    assert apply(y=None) == ERR
    assert apply(act=3) == ERR and "act=3" in _lib.last_error()
    assert apply(count=15.0) == ERR and "count" in _lib.last_error()      # fewer elements than this rank holds
    assert apply(count=float("nan")) == ERR
    assert apply(count=float("inf")) == ERR
    assert apply(sums=p + 4) == ERR and "8-byte" in _lib.last_error()
    assert apply(stats=p + 8) == ERR and "16-byte" in _lib.last_error()


def test_bn_train_bwd_validation():
    lib = _lib.lib
    raw, p = _buffers()
    ws = 1 << 20

    def bwd_stats(B=2, C_=4, P=8, z=p, g=p, stats=p, sums=p, act=1, nbytes=ws):
        return lib.ffb6d_bn_train_bwd_stats(z, g, stats, B, C_, P, act, 0.0, sums, p, p, p, nbytes, None)

    assert bwd_stats(B=0) == ERR and "bad size" in _lib.last_error()
    assert bwd_stats(C_=70000) == ERR
    assert bwd_stats(g=None) == ERR and "null" in _lib.last_error()
    assert bwd_stats(sums=None) == ERR
    assert bwd_stats(stats=None) == ERR
    assert bwd_stats(act=-1) == ERR
    assert bwd_stats(sums=p + 4) == ERR and "8-byte" in _lib.last_error()
    assert bwd_stats(stats=p + 4) == ERR and "16-byte" in _lib.last_error()
    assert bwd_stats(nbytes=8) == ERR and "workspace" in _lib.last_error()

    def bwd_apply(B=2, C_=4, P=8, z=p, g=p, stats=p, sums=p, count=16.0, act=1, dz=p):
        return lib.ffb6d_bn_train_bwd_apply(z, g, stats, sums, count, B, C_, P, act, 0.0, dz, None)

    assert bwd_apply(P=-1) == ERR and "bad size" in _lib.last_error()
    assert bwd_apply(dz=None) == ERR and "null" in _lib.last_error()
    assert bwd_apply(sums=None) == ERR
    assert bwd_apply(count=15.0) == ERR and "count" in _lib.last_error()
    assert bwd_apply(count=0.0) == ERR
    assert bwd_apply(act=5) == ERR
    assert bwd_apply(stats=p + 4) == ERR
