"""CPU-only: the CUDA library builds, loads without a GPU, exports every symbol include/*.h declares,
and refuses to work (instead of falling back to a CPU path) when no device is present."""
import os
import re
import subprocess
import sys

import pytest

import bzip3_b200
from bzip3_b200 import build as bz_build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    bz_build.build()
    return bzip3_b200.lib()


def declared_symbols():
    names = []
    for h in ("libbz3.h", "bz3_b200.h"):
        text = open(os.path.join(ROOT, "include", h)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names += re.findall(r"BZIP3_API[^;(]*?\b(bz3_\w+)\s*\(", text)
    return sorted(set(names))


def test_every_declared_symbol_is_exported(L):
    names = declared_symbols()
    assert len(names) >= 14 + 10
    for required in ("bz3_version", "bz3_last_error", "bz3_strerror", "bz3_new", "bz3_free", "bz3_bound",
                     "bz3_compress", "bz3_decompress", "bz3_min_memory_needed", "bz3_encode_block",
                     "bz3_decode_block", "bz3_encode_blocks", "bz3_decode_blocks",
                     "bz3_orig_size_sufficient_for_decode"):
        assert required in names
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/ but not exported by libbzip3_b200.so"


def test_pure_host_helpers(L):
    assert L.bz3_version().startswith(b"1.5.2")
    for n in (0, 1, 49, 50, 1000, 268435456):
        assert L.bz3_bound(n) == n + n // 50 + 32
    assert L.bz3_min_memory_needed(1000) == 0
    # reference figure (src/libbz3.c:999-1022): sizeof(struct bz3_state) + sizeof(state) + bound + 4*(bound+128) + 1 MiB
    b = 65 * 1024 + 65 * 1024 // 50 + 32
    assert L.bz3_min_memory_needed(65 * 1024) == 48 + 149024 + b + 4 * (b + 128) + 4 * (1 << 18)
    from tests import refs
    # the reference's figures
    refs.check_answer("min_memory_needed", [L.bz3_min_memory_needed(bs) for bs in MIN_MEMORY_BLOCK_SIZES])
    assert L.bz3_new(1000) is None  # block size out of range never needs a device


MIN_MEMORY_BLOCK_SIZES = (1000, 65 * 1024, 1 << 20, 16 << 20, 256 << 20, 511 << 20, (511 << 20) + 1)


def test_no_device_means_failure_not_fallback(L):
    """In a child process that sees no device (CUDA_VISIBLE_DEVICES empty), so that it runs on GPU machines too."""
    script = ("import sys\n"
              "sys.path.insert(0, %r)\n"
              "import bzip3_b200\n"
              "L = bzip3_b200.lib()\n"
              "assert L.bz3_b200_device_count() == 0\n"
              "assert L.bz3_new(1 << 20) is None\n"
              "try:\n"
              "    bzip3_b200.Bz3State(1 << 20)\n"
              "except bzip3_b200.Bz3Error:\n"
              "    print('REFUSED')\n" % ROOT)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "REFUSED" in r.stdout, r.stdout + r.stderr
