"""CPU: the Python face of the sentence server (engine.TTSServer) rejects bad arguments before anything reaches the library, and its ctypes
records match the C structs of include/infernos_b200.h."""
import ctypes
import os
import re

import pytest
import torch

from infernos_b200 import _lib
from infernos_b200.engine import TTSServer, _TTSChunk, _TTSServerStats

HDR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "infernos_b200.h")


class _Tail:
    has_postnet = True
    lib = None


def _closed():
    s = TTSServer.__new__(TTSServer)
    s.h = None
    return s


@pytest.mark.parametrize("kw,msg", [(dict(law=7), "law"), (dict(depth=0), "depth"), (dict(depth=5), "depth"), (dict(minlenratio=-1.0), "minlenratio"),
                                    (dict(threshold=float("nan")), "threshold"), (dict(poll_capacity=0), "poll_capacity")])
def test_constructor_checks(kw, msg):
    with pytest.raises(RuntimeError, match=msg):
        TTSServer(_Tail(), None, None, **kw)


def test_constructor_needs_postnet_weights():
    t = _Tail()
    t.has_postnet = False
    with pytest.raises(RuntimeError, match="post-net"):
        TTSServer(t, None, None)


@pytest.mark.parametrize("ids,spk,tag,msg", [([], torch.zeros(512), 0, "at least one token"), ([1.5, 2.0], torch.zeros(512), 0, "integer"),
                                             ([[1, 2], [3, 4]], torch.zeros(512), 0, "1-D"), ([1, 2], torch.zeros(511), 0, "512"),
                                             ([1, 2], torch.zeros(512), -1, "unsigned"), ([1, 2], torch.zeros(512), 2 ** 64, "unsigned"),
                                             ([2 ** 31], torch.zeros(512), 0, "int32")])
def test_submit_checks(ids, spk, tag, msg):
    with pytest.raises(RuntimeError, match=msg):
        _closed().submit(ids, spk, tag)


def test_submit_many_lengths_and_closed_server():
    s = _closed()
    with pytest.raises(RuntimeError, match="same length"):
        s.submit_many([[1]], [torch.zeros(512)] * 2, [0])
    s.submit_many([], [], [])                                 # nothing to do
    with pytest.raises(RuntimeError, match="closed"):
        s.submit([4, 5], torch.zeros(512), 1)
    with pytest.raises(RuntimeError, match="closed"):
        s.poll()


def test_records_match_the_header():
    hdr = open(HDR).read()
    for name, cls in (("b2_tts_chunk", _TTSChunk), ("b2_tts_server_stats", _TTSServerStats)):
        body = re.sub(r"/\*.*?\*/", "", re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), hdr, re.S).group(1), flags=re.S)
        fields = []
        for line in body.split(";"):
            line = line.strip()
            if line:
                typ, names = line.split(None, 1)
                fields += [(n.strip(), typ) for n in names.split(",")]
        size = {"uint64_t": 8, "int64_t": 8, "int32_t": 4}
        assert [f for f, _ in fields] == [f for f, _ in cls._fields_]
        assert [size[t] for _, t in fields] == [ctypes.sizeof(t) for _, t in cls._fields_]
    for sym in ("b2_tts_server_create", "b2_tts_server_destroy", "b2_tts_server_submit", "b2_tts_server_poll", "b2_tts_server_flush",
                "b2_tts_server_get_stats"):
        assert sym in _lib.SIGNATURES and re.search(r"\b%s\(" % sym, hdr)
