"""CPU: TTSServer.cancel (b2_tts_server_cancel) checks its tags before anything reaches the library, the entry point is declared and bound,
and the library rejects a NULL server."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from infernos_b200 import _lib
from infernos_b200.engine import TTSServer

HDR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "infernos_b200.h")


def _closed():
    s = TTSServer.__new__(TTSServer)
    s.h = None
    return s


def test_cancel_is_declared_and_bound():
    assert _lib.SIGNATURES["b2_tts_server_cancel"] == (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int])
    assert re.search(r"\bb2_tts_server_cancel\(b2_tts_server \*s, const uint64_t \*tags, int n\);", open(HDR).read())


@pytest.mark.parametrize("tags", [-1, 2 ** 64, [1, -1], [2 ** 64], 1.5, [1, 2.0], np.float64(3.0), "7", [None], torch.tensor([1.0, 2.0])])
def test_cancel_rejects_bad_tags_before_the_library(tags):
    with pytest.raises(RuntimeError, match="unsigned 64-bit"):
        _closed().cancel(tags)


@pytest.mark.parametrize("tags", [0, 2 ** 64 - 1, [3, 3, 4], (5,), [], np.uint64(2 ** 63), torch.tensor([1, 2]), range(3)])
def test_cancel_on_a_closed_server_raises(tags):
    with pytest.raises(RuntimeError, match="closed"):
        _closed().cancel(tags)


def test_cancel_with_a_null_server_fails():
    from infernos_b200 import build
    build.build()
    lib = _lib.load()
    tg = (ctypes.c_uint64 * 1)(1)
    assert lib.b2_tts_server_cancel(None, tg, 1) < 0
    assert b"null server" in lib.b2_last_error(None)
