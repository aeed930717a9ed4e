"""uqs_replay_recentering_dev without a device: the symbol is exported and every call, well-formed or not, returns
UQS_ERR_NOT_INIT (there is no CPU implementation to fall back to)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_symbol_is_exported(pkg):
    assert "uqs_replay_recentering_dev" in pkg.exported_symbols()
    out = subprocess.check_output(["nm", "-D", "--defined-only", pkg.LIB_PATH], text=True)
    assert " T uqs_replay_recentering_dev" in out and " T uqs_replay_recentering" in out


def test_calls_fail_without_a_device(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.UqsError):
        pkg.init(0)
    p = pkg.make_params(400, 400, 0.05, size_m=20.0)
    L = pkg.lib()
    st = pkg.Stats()
    good = [ctypes.c_void_p(16)] * 8
    for F, N, bufs, cap in [(2, 10, good, 0), (0, 10, good, 0), (2, -1, good, 0), (2, 10, [None] * 8, 0), (2, 10, good, -1),
                            (2, 10, good[:7] + [None], 4)]:
        rc = L.uqs_replay_recentering_dev(ctypes.byref(p), F, N, *bufs, cap, ctypes.byref(st))
        assert rc == pkg.ERR_NOT_INIT, (F, N, cap)
    z = np.zeros((2, 10), np.float32)
    with pytest.raises(pkg.UqsError) as e:
        pkg.replay_recentering(p, z[0], z[0], z[0], np.zeros((10, 32), np.float32))
    assert e.value.code == pkg.ERR_NOT_INIT
