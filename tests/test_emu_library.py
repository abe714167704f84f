"""The WHOLE library on the CPU thread-block emulator: bzip3_b200/csrc/bz3_api.cu -- the C ABI, the block framing and
validation, every launch sequence and every kernel -- compiled by g++ on top of tests/native/cta_emu.h into
tests/_build/libbzip3_emu.so and driven through the same Python binding as the GPU library.

Test infrastructure: it lets the "no GPU" suite check the product's host logic and kernels against the oracle on small
inputs (the emulator codes a few kilobytes per second).  The GPU parity tests remain the gate for the real library;
what runs here is the same source, not the same binary."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import bzip3_b200
from bzip3_b200 import synth
from tests import refs
from tests.test_oracle import hostile_variants

ROOT = refs.ROOT
SO = os.path.join(ROOT, "tests", "_build", "libbzip3_emu.so")
CSRC = os.path.join(ROOT, "bzip3_b200", "csrc")
EMU_H = os.path.join(ROOT, "tests", "native", "cta_emu.h")
SRCS = [os.path.join(CSRC, "bz3_api.cu"), os.path.join(ROOT, "tests", "native", "cta_emu.cpp")]
BS = 65 * 1024 + 1024   # smallest legal block size is 65 KiB (src/libbz3.c:536)
CUT = 1400              # bytes per case: the emulated suffix sort does ~3 KB/s


def build_emulated_library():
    deps = SRCS + [EMU_H] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(ROOT, "include", "libbz3.h"), os.path.join(ROOT, "include", "bz3_b200.h")]
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-DBZ_EMU", "-include",
                               EMU_H, "-x", "c++", "-o", SO] + SRCS + ["-lpthread"])
    return SO


@pytest.fixture(scope="module")
def emulib():
    """Points the Python binding at the emulated library for the tests of this module, then restores it."""
    so = build_emulated_library()
    saved = (bzip3_b200.LIB_PATH, bzip3_b200._lib)
    bzip3_b200.LIB_PATH, bzip3_b200._lib = so, None
    try:
        yield bzip3_b200.lib()
    finally:
        bzip3_b200.LIB_PATH, bzip3_b200._lib = saved


@pytest.fixture(scope="module")
def st(emulib):
    with bzip3_b200.Bz3State(BS) as s:
        yield s


CASES = [(name, bytes(d[:CUT])) for name, d in synth.edge_cases()]
IDS = [c[0] for c in CASES]


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_block_roundtrip_vs_oracle(st, name, data):
    enc_o, r_o, e_o = refs.oracle_encode_block(data, BS)
    enc_g, r_g = st.encode_block(data)
    assert r_g == r_o, (r_g, r_o, st.last_error)
    if len(data) >= 64:
        assert st.last_error == e_o
    assert enc_g == enc_o
    dec, r = st.decode_block(enc_o, len(data))
    assert r == len(data) and dec == data
    if len(data) >= 64:
        assert st.last_error == 0


def test_block_too_big_and_raw_paths(st):
    enc, r = st.encode_block(bytes(BS + 1))
    assert r == -1 and st.last_error == bzip3_b200.BZ3_ERR_DATA_TOO_BIG
    enc, r = st.encode_block(b"tiny")  # the reference returns early without touching last_error (src/libbz3.c:596-601)
    assert r == 12 and st.last_error == bzip3_b200.BZ3_ERR_DATA_TOO_BIG
    dec, r = st.decode_block(enc, 4)
    assert dec == b"tiny" and st.last_error == bzip3_b200.BZ3_ERR_DATA_TOO_BIG


@pytest.mark.parametrize("name", ["raw63", "coded65_text", "random_10k", "escape_heavy"])
def test_hostile_decode_error_parity(st, name):
    """Truncated, bit-flipped and header-patched blocks: same return value, error number and bytes as the oracle."""
    data = dict(CASES)[name][:1200]
    enc, r, e = refs.oracle_encode_block(data, BS)
    rng = np.random.default_rng(len(data))
    for k, (venc, osz, bsz, csz) in enumerate(hostile_variants(enc, len(data), BS, rng)):
        want = refs.oracle_decode_block(venc, osz, BS, buffer_size=bsz, compressed_size=csz, err_init=55)
        got_bytes, got_r = st.decode_block(venc, osz, buffer_size=bsz, compressed_size=csz)
        assert got_r == want[1], (name, k, got_r, want[1:], st.last_error)
        if want[2] != 55:  # the oracle wrote an error code
            assert st.last_error == want[2], (name, k, st.last_error, want[2])
        if got_r >= 0:
            assert got_bytes == want[0], (name, k)


def test_batch_api_uses_threads_and_matches_single_blocks(emulib):
    L = emulib
    datas = [synth.zipf_text(1500, seed=5).tobytes(), synth.log_stream(1200, seed=6).tobytes(), b"short",
             bytes(np.random.default_rng(3).integers(0, 256, 900, dtype=np.uint8))]
    states = [bzip3_b200.Bz3State(BS) for _ in datas]
    try:
        bufs = []
        for d in datas:
            b = np.zeros(bzip3_b200.bound(BS) + 64, np.uint8)
            b[:len(d)] = np.frombuffer(d, np.uint8)
            bufs.append(b)
        sizes = [len(d) for d in datas]
        out_sizes = bzip3_b200.encode_blocks(states, bufs, sizes)
        for d, b, r in zip(datas, bufs, out_sizes):
            enc_o, r_o, _ = refs.oracle_encode_block(d, BS)
            assert r == r_o and bytes(b[:r]) == enc_o
        errs = bzip3_b200.decode_blocks(states, bufs, [len(b) for b in bufs], out_sizes, sizes)
        for d, b, e in zip(datas, bufs, errs):
            assert e == 0 and bytes(b[:len(d)]) == d
    finally:
        for s in states:
            s.close()


def test_frame_api_and_helpers(emulib):
    L = emulib
    data = synth.zipf_text(2200, seed=9)
    n = len(data)
    cap = bzip3_b200.bound(n) + 64
    out = np.zeros(cap, np.uint8)
    osz = C.c_size_t(cap)
    assert L.bz3_compress(BS, refs.ptr(data), refs.ptr(out), n, C.byref(osz)) == 0
    frame = out[:osz.value].copy()
    assert bytes(frame[:5]) == b"BZ3v1"
    back = np.zeros(n + 64, np.uint8)
    bsz = C.c_size_t(n + 64)
    assert L.bz3_decompress(refs.ptr(frame), refs.ptr(back), len(frame), C.byref(bsz)) == 0
    assert bsz.value == n and bytes(back[:n]) == bytes(data)
    refs.check_answer("frame/zipf2200_seed9", [len(frame), refs.digest(frame)])   # the same frame from the reference
    assert L.bz3_bound(1000) == 1000 + 1000 // 50 + 32
    assert not L.bz3_new(1000) and not L.bz3_new((511 << 20) + 1)   # block size out of range


def test_stage_workspaces_are_shared_by_the_states_of_a_device(emulib, st):
    """The 48 B/B scratch of mRLE / suffix sort / inverse BWT is a per-device pool leased per stage call (ArenaPool in
    bz3_api.cu), not a per-state allocation: what a state owns is three block buffers and the LZP table."""
    L = emulib
    base = L.bz3_b200_workspace_bytes(st.handle)
    own = L.bz3_b200_device_bytes(st.handle)
    assert 0 < own < 3.2 * bzip3_b200.bound(BS) + (1 << 20) + 4096
    assert base >= 48 * BS
    with bzip3_b200.Bz3State(BS) as s2:    # from the second state on there are two (BZ3_B200_ARENAS), and never more
        two = L.bz3_b200_workspace_bytes(s2.handle)
        assert 2 * 48 * BS <= two < 2 * 52 * BS and two in (base, 2 * base)   # (earlier tests may have had two states already)
        with bzip3_b200.Bz3State(BS) as s2b:
            assert L.bz3_b200_workspace_bytes(s2b.handle) == two
        with bzip3_b200.Bz3State(4 * BS) as s3:   # a larger one grows the shared workspaces
            grown = L.bz3_b200_workspace_bytes(s3.handle)
            assert grown >= 2 * 48 * 4 * BS and L.bz3_b200_workspace_bytes(st.handle) == grown
            data = synth.zipf_text(1300, seed=11).tobytes()
            want = refs.oracle_encode_block(data, 4 * BS)
            enc, r = s3.encode_block(data)
            assert r == want[1] and enc == want[0]
        data = synth.log_stream(1300, seed=12).tobytes()   # the smaller states keep working in the grown workspaces
        want = refs.oracle_encode_block(data, BS)
        enc, r = s2.encode_block(data)
        assert r == want[1] and enc == want[0]
        dec, r = st.decode_block(enc, len(data))
        assert r == len(data) and dec == data


def test_one_workspace_serves_a_batch_of_blocks(emulib):
    """BZ3_B200_ARENAS=1: the host threads of bz3_encode_blocks / bz3_decode_blocks queue for the only workspace."""
    import subprocess
    import sys
    script = (
        "import sys\n"
        "sys.path.insert(0, %r)\n"
        "import numpy as np\n"
        "import bzip3_b200\n"
        "from bzip3_b200 import synth\n"
        "from tests import refs\n"
        "bs = %d\n"
        "datas = [synth.zipf_text(900 + 100 * k, seed=k).tobytes() for k in range(5)]\n"
        "states = [bzip3_b200.Bz3State(bs) for _ in datas]\n"
        "L = states[0].L\n"
        "print('WORKSPACE', L.bz3_b200_workspace_bytes(states[0].handle) // (48 * bs))\n"
        "bufs = []\n"
        "for d in datas:\n"
        "    b = np.zeros(bzip3_b200.bound(bs) + 64, np.uint8)\n"
        "    b[:len(d)] = np.frombuffer(d, np.uint8)\n"
        "    bufs.append(b)\n"
        "sizes = [len(d) for d in datas]\n"
        "out = bzip3_b200.encode_blocks(states, bufs, sizes)\n"
        "ok = all(bytes(b[:r]) == refs.oracle_encode_block(d, bs)[0] for d, b, r in zip(datas, bufs, out))\n"
        "errs = bzip3_b200.decode_blocks(states, bufs, [len(b) for b in bufs], out, sizes)\n"
        "ok = ok and all(e == 0 and bytes(b[:len(d)]) == d for d, b, e in zip(datas, bufs, errs))\n"
        "for s in states: s.close()\n"
        "with bzip3_b200.Bz3State(bs) as s:\n"
        "    ok = ok and s.encode_block(datas[0])[0] == refs.oracle_encode_block(datas[0], bs)[0]\n"
        "print('EXACT', ok)\n" % (ROOT, BS))
    env = dict(os.environ, BZ3_B200_LIB=SO, BZ3_B200_ARENAS="1")
    out = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=900)
    assert "WORKSPACE 1" in out.stdout, out.stdout + out.stderr
    assert "EXACT True" in out.stdout, out.stdout + out.stderr


def test_out_of_device_memory_is_reported_by_bz3_new_and_spares_the_live_states(emulib):
    """A state whose workspace does not fit makes bz3_new return NULL (as the reference's does on a failed malloc,
    src/libbz3.c:553-561); the states that already exist keep their workspaces and keep coding."""
    import subprocess
    import sys
    script = (
        "import sys\n"
        "sys.path.insert(0, %r)\n"
        "import bzip3_b200\n"
        "from bzip3_b200 import synth\n"
        "from tests import refs\n"
        "bs = %d\n"
        "L = bzip3_b200.lib()\n"
        "a = bzip3_b200.Bz3State(bs)\n"
        "lone = L.bz3_b200_workspace_bytes(a.handle)\n"
        "b = bzip3_b200.Bz3State(bs)\n"
        "before = L.bz3_b200_workspace_bytes(a.handle)\n"
        "print('LONE', 48 * bs <= lone < 52 * bs, before == 2 * lone)\n"
        "print('BIG', L.bz3_new(8 * bs))\n"
        "print('SAME', L.bz3_b200_workspace_bytes(a.handle) == before)\n"
        "data = synth.zipf_text(1000, seed=4).tobytes()\n"
        "want = refs.oracle_encode_block(data, bs)\n"
        "ok = True\n"
        "for s in (a, b):\n"
        "    enc, r = s.encode_block(data)\n"
        "    dec, r2 = s.decode_block(enc, len(data))\n"
        "    ok = ok and r == want[1] and enc == want[0] and dec == data\n"
        "print('EXACT', ok)\n" % (ROOT, BS))
    cap = 48 * 3 * BS   # enough for the workspace of a BS state (and for block buffers), not for an 8 * BS state
    env = dict(os.environ, BZ3_B200_LIB=SO, BZ_EMU_MALLOC_MAX=str(cap))
    out = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=900)
    assert "LONE True True" in out.stdout, out.stdout + out.stderr   # a lone state gets one workspace, the second state the second
    assert "BIG None" in out.stdout, out.stdout + out.stderr
    assert "SAME True" in out.stdout and "EXACT True" in out.stdout, out.stdout + out.stderr
