"""C-ABI surface (no GPU needed): the library builds for sm_100a, loads, and exports every symbol the header declares."""
import ctypes
import os
import re

import pytest

import spark_s3_shuffle_b200 as pkg
from without_gpu import rerun_without_gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "b200shuffle.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b2s_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_every_declared_symbol():
    path = pkg.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    syms = _header_symbols()
    assert len(syms) >= 25
    for s in syms:
        assert hasattr(lib, s), "libb200shuffle.so does not export %s" % s


def test_python_prototypes_cover_the_header():
    assert sorted(pkg.capi.SYMBOLS) == _header_symbols()


def test_sm100a_cubin_is_embedded():
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", pkg.lib_path()], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_strerror_and_bounds_need_no_device():
    c = pkg.capi
    L = c.load()
    assert L.b2s_strerror(c.E_CORRUPT) == b"Stream is corrupted"
    assert L.b2s_strerror(c.E_CHECKSUM).startswith(b"Invalid checksum detected")
    assert c.compress_bound(c.CODEC_LZ4BLOCK, 0, 0) == 21          # empty stream = end mark only
    assert c.compress_bound(c.CODEC_LZ4BLOCK, 32768, 65537) == 65537 + 4 * 21
    assert L.b2s_version() == 0x000100


def test_fails_loudly_without_a_gpu():
    """No CPU fallback: on a box without CUDA devices init (and therefore every compute call) reports B2S_E_CUDA."""
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = os.path.exists("/dev/nvidia0")
    if has_gpu:
        rerun_without_gpu(__file__, "test_fails_loudly_without_a_gpu")
        return
    c = pkg.capi
    L = c.load()
    assert L.b2s_init(0, 0, 0) == c.E_CUDA
    assert L.b2s_device_count() == c.E_NOT_INIT
    with pytest.raises(c.B2SError):
        c.checksum_batch(c.CHECKSUM_CRC32, [b"abc"])
