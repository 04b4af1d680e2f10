"""Helpers for the WAV format tests: ctypes wrappers of the checker's WAV sample codecs, an independent RIFF chunk walker,
and a builder for headers that Python's own writers do not produce (WAVE_FORMAT_EXTENSIBLE, unusual tags, extra chunks)."""
import ctypes
import hashlib
import os
import struct
import subprocess
import tempfile

import numpy as np

# libsndfile's sub-type codes, as include/flan_b200.h carries them (FLAN_B200_WAV_*)
PCM_16, PCM_24, PCM_32, PCM_U8, FLOAT, DOUBLE = 0x2, 0x3, 0x4, 0x5, 0x6, 0x7
ALL = [PCM_U8, PCM_16, PCM_24, PCM_32, FLOAT, DOUBLE]
WIDTH = {PCM_U8: 1, PCM_16: 2, PCM_24: 3, PCM_32: 4, FLOAT: 4, DOUBLE: 8}
NAME = {PCM_U8: "PCM_U8", PCM_16: "PCM_16", PCM_24: "PCM_24", PCM_32: "PCM_32", FLOAT: "FLOAT", DOUBLE: "DOUBLE"}

# KSDATAFORMAT_SUBTYPE_PCM / _IEEE_FLOAT: the format tag, then this fixed tail
GUID_TAIL = bytes([0x00, 0x00, 0x00, 0x00, 0x10, 0x00, 0x80, 0x00, 0x00, 0xAA, 0x00, 0x38, 0x9B, 0x71])


WAV_ORACLE_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "wav_oracle.c")


def wav_oracle_lib():
    """tests/cpp/wav_oracle.c built as the oracle's Makefile builds pv_oracle.c (gcc -O2 -ffp-contract=off), into the
    temporary directory: the repository tree is left as it is. The file name carries a hash of the source."""
    src = open(WAV_ORACLE_SRC, "rb").read()
    path = os.path.join(tempfile.gettempdir(), "flan_b200_wav_oracle_%d_%s.so" % (os.getuid(), hashlib.sha256(src).hexdigest()[:16]))
    if not os.path.exists(path):
        tmp = path + ".%d.tmp" % os.getpid()
        subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-std=c11", "-shared", "-o", tmp, WAV_ORACLE_SRC, "-lm"],
                       check=True)
        os.replace(tmp, path)
    return path


class OracleWav:
    """The checker's WAV sample codecs (tests/cpp/wav_oracle.c). `base` is the oracle_lib.Oracle whose PCM-24 restatement
    (pvo_pcm24_*) the PCM_24 case is compared with."""

    def __init__(self, base):
        L = ctypes.CDLL(wav_oracle_lib())
        fp, bp = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint8)
        L.wavo_pcm_width.argtypes = [ctypes.c_int]
        L.wavo_pcm_encode.argtypes = [fp, ctypes.c_int, ctypes.c_int64, ctypes.c_int, bp]
        L.wavo_pcm_decode.argtypes = [bp, ctypes.c_int, ctypes.c_int64, ctypes.c_int, fp]
        self.L, self.base, self._fp, self._bp = L, base, fp, bp

    def pcm_width(self, subtype):
        return int(self.L.wavo_pcm_width(subtype))

    def pcm_encode(self, audio, subtype):
        """planar float32 [C, n] -> interleaved sample bytes of a WAV sub-type (libsndfile's code)."""
        audio = np.ascontiguousarray(audio, np.float32)
        C, n = audio.shape
        out = np.empty(C * n * self.pcm_width(subtype), np.uint8)
        assert self.L.wavo_pcm_encode(audio.ctypes.data_as(self._fp), C, n, subtype, out.ctypes.data_as(self._bp)) == 0
        return out

    def pcm_decode(self, data, C, n, subtype):
        data = np.ascontiguousarray(data, np.uint8)
        assert data.size >= C * n * self.pcm_width(subtype)
        out = np.empty((C, n), np.float32)
        assert self.L.wavo_pcm_decode(data.ctypes.data_as(self._bp), C, n, subtype, out.ctypes.data_as(self._fp)) == 0
        return out


def chunks(raw):
    """[(id, payload offset, size)] of a RIFF/WAVE file's top-level chunks."""
    assert raw[:4] == b"RIFF" and raw[8:12] == b"WAVE"
    out, pos = [], 12
    while pos + 8 <= len(raw):
        cid, size = raw[pos:pos + 4], struct.unpack("<I", raw[pos + 4:pos + 8])[0]
        out.append((cid, pos + 8, size))
        pos += 8 + size + (size & 1)
    return out


def chunk(raw, cid):
    for c, off, size in chunks(raw):
        if c == cid:
            return raw[off:off + size]
    return None


def fmt_fields(raw):
    """(tag, channels, rate, byte rate, block align, bits) of the fmt chunk."""
    return struct.unpack("<HHIIHH", chunk(raw, b"fmt ")[:16])


def data_bytes(path):
    with open(path, "rb") as f:
        return np.frombuffer(chunk(f.read(), b"data"), np.uint8)


def build_wav(data, C, sr, tag, bits, block=None, extensible=False, valid_bits=None, sub_tail=GUID_TAIL, before_data=()):
    """A WAVE file's bytes. extensible: tag 0xFFFE with `tag` as the sub-format's first two bytes. before_data: extra
    (id, payload) chunks placed between fmt and data (odd sizes get their pad byte)."""
    block = block if block is not None else C * ((bits + 7) // 8)
    fmt = struct.pack("<HHIIHH", 0xFFFE if extensible else tag, C, sr, sr * block, block, bits)
    if extensible:
        fmt += struct.pack("<HHI", 22, valid_bits or bits, 0) + struct.pack("<H", tag) + sub_tail
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt
    for cid, payload in before_data:
        body += cid + struct.pack("<I", len(payload)) + payload + (b"\0" if len(payload) & 1 else b"")
    data = bytes(data)
    body += b"data" + struct.pack("<I", len(data)) + data + (b"\0" if len(data) & 1 else b"")
    return b"RIFF" + struct.pack("<I", len(body)) + body


def interleave(values):
    """Planar [C, n] -> interleaved [n * C]."""
    return np.ascontiguousarray(np.asarray(values).T).reshape(-1)
