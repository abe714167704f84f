"""The container front end with the deep block queue (bz3_b200_encode_fd / bz3_b200_decode_fd, csrc/stream.h) on the GPU:
more blocks than queue slots, several blocks in flight, bytes compared with the reference tool's container built around
the oracle's blocks (and with what the reference binary wrote, tests/golden/reference_answers.json)."""
import ctypes as C
import os
import struct
import subprocess

import pytest

import bzip3_b200
from bzip3_b200 import synth
from tests import refs

pytestmark = pytest.mark.gpu
BS = 1 << 20


def container(data, bs):
    out = bytearray(b"BZ3v1" + struct.pack("<i", bs))
    for at in range(0, len(data), bs):
        blk = data[at:at + bs]
        enc, r, _ = refs.oracle_encode_block(blk, bs)
        out += struct.pack("<ii", r, len(blk)) + enc[:r]
    return bytes(out)


def corpus_data():
    return (synth.zipf_text(2_300_000, seed=21).tobytes() + bytes(300_000) + synth.log_stream(1_900_000, seed=22).tobytes()
            + synth.source_corpus(1_200_000, seed=23).tobytes() + b"end")


@pytest.fixture(scope="module")
def corpus():
    data = corpus_data()
    return data, container(data, BS)


def run_fd(fn, src_bytes, tmp_path, *args, test_only=False):
    src, dst = tmp_path / "in", tmp_path / "out"
    src.write_bytes(src_bytes)
    fi = os.open(src, os.O_RDONLY)
    fo = -1 if test_only else os.open(dst, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
    nin, nout = C.c_uint64(0), C.c_uint64(0)
    try:
        rc = fn(fi, fo, *args, C.byref(nin), C.byref(nout))
    finally:
        os.close(fi)
        if fo >= 0:
            os.close(fo)
    return rc, (b"" if test_only else dst.read_bytes()), nin.value, nout.value


@pytest.mark.parametrize("depth", [1, 4, 0])
def test_stream_roundtrip_bytes(tmp_path, corpus, depth):
    L = bzip3_b200.lib()
    data, want = corpus
    rc, got, nin, nout = run_fd(L.bz3_b200_encode_fd, data, tmp_path, BS, depth)
    assert rc == 0 and nin == len(data) and nout == len(want)
    assert got == want
    rc, back, nin, nout = run_fd(L.bz3_b200_decode_fd, want, tmp_path, depth)
    assert rc == 0 and back == data
    rc, _, _, nout = run_fd(L.bz3_b200_decode_fd, want, tmp_path, depth, test_only=True)
    assert rc == 0 and nout == len(data)


def test_stream_damaged_block(tmp_path, corpus):
    L = bzip3_b200.lib()
    data, want = corpus
    at = 9
    c0 = struct.unpack_from("<i", want, at)[0]
    second = at + 8 + c0
    c1, o1 = struct.unpack_from("<ii", want, second)
    bad = bytearray(want)
    bad[second + 8 + c1 // 3] ^= 0x04
    expect = refs.oracle_decode_block(bytes(bad[second + 8: second + 8 + c1]), o1, BS, err_init=55)
    rc, back, _, _ = run_fd(L.bz3_b200_decode_fd, bytes(bad), tmp_path, 3)
    assert expect[1] == -1 and rc == expect[2]
    assert back == data[:BS]          # the block before the damaged one is out, nothing after it
    rc, back, _, _ = run_fd(L.bz3_b200_decode_fd, want[:second + 8 + c1 // 2], tmp_path, 3)
    assert rc == -23 and back == data[:BS]


def test_command_line_tool(tmp_path, corpus):
    cli = os.path.join(refs.ROOT, "bzip3_b200", "bz3b200")
    if not (os.path.exists(cli) and os.access(cli, os.X_OK)):
        pytest.skip("bzip3_b200/bz3b200 not built")
    data, want = corpus
    r = subprocess.run([cli, "-e", "-b", "1", "-j", "5"], input=data, capture_output=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert r.stdout == want
    # what `bzip3 -e -b 1 -j 4` writes for the same input; the reference decodes that file to the input
    refs.check_answer("cli/stream_corpus_b1", [len(r.stdout), refs.digest(r.stdout)])
    r = subprocess.run([cli, "-d", "-j", "3"], input=want, capture_output=True, timeout=600)
    assert r.returncode == 0 and r.stdout == data


def many_blocks_check(L, bs, nblk, nbytes):
    import numpy as np
    gens = (synth.zipf_text, synth.log_stream, synth.source_corpus)
    datas = [gens[k % 3](nbytes - (nbytes // 256) * (k % 5), seed=100 + k).tobytes() for k in range(nblk)]
    states = [bzip3_b200.Bz3State(bs) for _ in datas]
    try:
        ws = L.bz3_b200_workspace_bytes(states[0].handle)
        own = L.bz3_b200_device_bytes(states[0].handle)
        assert 2 * 48 * bs <= ws < 2 * 56 * bs and own < 3.3 * bzip3_b200.bound(bs) + (2 << 20)
        bufs = []
        for d in datas:
            b = np.zeros(bzip3_b200.bound(bs) + 64, np.uint8)
            b[:len(d)] = np.frombuffer(d, np.uint8)
            bufs.append(b)
        sizes = bzip3_b200.encode_blocks(states, bufs, [len(d) for d in datas])
        assert all(s.last_error == 0 for s in states)
        for k in range(0, nblk, 5):
            assert bytes(bufs[k][:sizes[k]]) == refs.oracle_encode_block(datas[k], bs)[0], k
        bzip3_b200.decode_blocks(states, bufs, [len(b) for b in bufs], sizes, [len(d) for d in datas])
        for d, b, s in zip(datas, bufs, states):
            assert s.last_error == 0 and bytes(b[:len(d)]) == d
        assert L.bz3_b200_workspace_bytes(states[0].handle) == ws
    finally:
        for s in states:
            s.close()


def test_many_blocks_in_flight_share_two_workspaces():
    """48 states / streams at once (more than the 32 hardware queues), all leasing the device's two stage workspaces:
    bit-exact against the oracle, and the device footprint is 48 small states + 2 workspaces, not 48 workspaces."""
    many_blocks_check(bzip3_b200.lib(), 256 << 10, 48, (256 << 10) - 8)


def test_stream_over_all_visible_gpus(tmp_path, corpus):
    """devices = 0: the workers are dealt over every visible GPU of this process (one GPU on a single-GPU box, where this
    equals the plain call); the bytes do not depend on where a block was coded."""
    L = bzip3_b200.lib()
    data, want = corpus
    rc, got, _, _ = run_fd(L.bz3_b200_encode_fd2, data, tmp_path, BS, 6, 0)
    assert rc == 0 and got == want
    rc, back, _, _ = run_fd(L.bz3_b200_decode_fd2, want, tmp_path, 6, 0)
    assert rc == 0 and back == data


def test_mutated_containers_follow_the_reference_loop(tmp_path, corpus):
    """Random damage to the container: same verdict and same bytes out as the reference tool's loop (the model of
    tests/test_emu_stream.py, which is pinned on the reference binary in the CPU suite)."""
    import numpy as np
    from tests.test_emu_stream import reference_loop_model
    L = bzip3_b200.lib()
    data, good = corpus
    small = good[: 9]
    at = 9
    for _ in range(3):   # the first three blocks are enough: three CPU oracle decodes per trial
        c = struct.unpack_from("<i", good, at)[0]
        small += good[at: at + 8 + c]
        at += 8 + c
    rng = np.random.default_rng(7)
    for trial in range(10):
        blob = bytearray(small)
        kind = trial % 5
        if kind == 0:
            blob[int(rng.integers(30, len(blob)))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1:
            blob = blob[: int(rng.integers(9, len(blob)))]
        elif kind == 2:
            blob[9 + int(rng.integers(0, 17))] ^= int(rng.integers(1, 256))
        elif kind == 3:
            blob[int(rng.integers(0, 9))] ^= int(rng.integers(1, 256))
        else:
            blob += bytes(rng.integers(0, 256, int(rng.integers(1, 12)), dtype=np.uint8))
        blob = bytes(blob)
        want = reference_loop_model(blob, BS)
        rc, back, _, _ = run_fd(L.bz3_b200_decode_fd, blob, tmp_path, 1 + trial % 3)
        assert rc == want[0], (trial, kind, rc, want[0])
        assert back == want[1], (trial, kind, len(back), len(want[1]))
