"""The container front end with the deep block queue (bz3_b200_encode_fd / bz3_b200_decode_fd, csrc/stream.h; SURVEY 8 f2)
on the emulator build of the library: the bytes must be those of the reference's command line tool -- rebuilt here from
the container layout of src/main.c:171-278 around the oracle's blocks, and compared with what the reference binary itself
wrote (tests/golden/reference_answers.json) -- for several blocks in flight, through files and pipes, and every error path
must wind the reader / workers / writer down without a hang."""
import ctypes as C
import os
import struct
import subprocess
import threading

import numpy as np
import pytest

import bzip3_b200
from bzip3_b200 import synth
from tests import refs
from tests.test_emu_library import BS, build_emulated_library


@pytest.fixture(scope="module")
def L():
    so = build_emulated_library()
    saved = (bzip3_b200.LIB_PATH, bzip3_b200._lib)
    bzip3_b200.LIB_PATH, bzip3_b200._lib = so, None
    try:
        yield bzip3_b200.lib()
    finally:
        bzip3_b200.LIB_PATH, bzip3_b200._lib = saved


def squeezable(nbytes, seed):
    """Data that LZP and mRLE shrink to a few hundred bytes per block, so that the emulated suffix sort stays cheap."""
    rng = np.random.default_rng(seed)
    line = synth.log_stream(300, seed=seed).tobytes()
    out = bytearray()
    while len(out) < nbytes:
        out += line
        if rng.integers(0, 4) == 0:
            out += bytes([int(rng.integers(32, 127))]) * int(rng.integers(3, 200))
    return bytes(out[:nbytes])


def container(data, bs):
    """What `bzip3 -e` writes for `data` with block size `bs` (src/main.c:171-203, :231-251)."""
    out = bytearray(b"BZ3v1" + struct.pack("<i", bs))
    for at in range(0, len(data), bs):
        blk = data[at:at + bs]
        enc, r, _ = refs.oracle_encode_block(blk, bs)
        out += struct.pack("<ii", r, len(blk)) + enc[:r]
    return bytes(out)


def encode_file(L, tmp_path, data, bs, depth, name="in"):
    src, dst = tmp_path / (name + ".bin"), tmp_path / (name + ".bz3")
    src.write_bytes(data)
    fi, fo = os.open(src, os.O_RDONLY), os.open(dst, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
    try:
        nin, nout = C.c_uint64(0), C.c_uint64(0)
        rc = L.bz3_b200_encode_fd(fi, fo, bs, depth, C.byref(nin), C.byref(nout))
    finally:
        os.close(fi)
        os.close(fo)
    return rc, dst.read_bytes(), nin.value, nout.value


def decode_bytes(L, tmp_path, blob, depth, test_only=False, name="x"):
    src, dst = tmp_path / (name + ".in.bz3"), tmp_path / (name + ".out")
    src.write_bytes(blob)
    fi = os.open(src, os.O_RDONLY)
    fo = -1 if test_only else os.open(dst, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
    try:
        nin, nout = C.c_uint64(0), C.c_uint64(0)
        rc = L.bz3_b200_decode_fd(fi, fo, depth, C.byref(nin), C.byref(nout))
    finally:
        os.close(fi)
        if fo >= 0:
            os.close(fo)
    return rc, (b"" if test_only else dst.read_bytes()), nin.value, nout.value


@pytest.fixture(scope="module")
def four_blocks():
    data = squeezable(3 * BS + 7000, seed=5)
    return data, container(data, BS)


@pytest.mark.parametrize("depth", [2, 6])
def test_container_bytes_equal_the_reference_layout(L, tmp_path, four_blocks, depth):
    data, want = four_blocks
    rc, got, nin, nout = encode_file(L, tmp_path, data, BS, depth)
    assert rc == 0 and got == want
    assert nin == len(data) and nout == len(want)
    rc, back, nin, nout = decode_bytes(L, tmp_path, want, depth)
    assert rc == 0 and back == data and nin == len(want) and nout == len(data)
    rc, _, _, nout = decode_bytes(L, tmp_path, want, depth, test_only=True)
    assert rc == 0 and nout == len(data)


def test_pipes_and_short_reads(L, four_blocks):
    """Input arriving in small pieces through a pipe fills the blocks exactly like a file (fread semantics, :236)."""
    data, want = four_blocks
    ri, wi = os.pipe()
    ro, wo = os.pipe()
    got = bytearray()

    def feed():
        for at in range(0, len(data), 5000):
            os.write(wi, data[at:at + 5000])
        os.close(wi)

    def drain():
        while True:
            b = os.read(ro, 65536)
            if not b:
                break
            got.extend(b)

    tf, td = threading.Thread(target=feed), threading.Thread(target=drain)
    tf.start()
    td.start()
    rc = L.bz3_b200_encode_fd(ri, wo, BS, 2, None, None)
    os.close(wo)
    os.close(ri)
    tf.join()
    td.join()
    os.close(ro)
    assert rc == 0 and bytes(got) == want


def test_empty_and_tiny_inputs(L, tmp_path):
    rc, got, nin, nout = encode_file(L, tmp_path, b"", BS, 3, "empty")
    assert rc == 0 and got == b"BZ3v1" + struct.pack("<i", BS) and nout == 9   # no block at all, :237
    rc, back, _, _ = decode_bytes(L, tmp_path, got, 3, name="empty")
    assert rc == 0 and back == b""
    for data in (b"a", bytes(range(63)), synth.zipf_text(700, seed=1).tobytes()):   # raw (<64 B) and coded single blocks
        rc, got, _, _ = encode_file(L, tmp_path, data, BS, 2, "tiny")
        assert rc == 0 and got == container(data, BS)
        rc, back, _, _ = decode_bytes(L, tmp_path, got, 2, name="tiny")
        assert rc == 0 and back == data


def test_against_the_reference_binary(L, tmp_path):
    """The file `bzip3 -e -b 1` writes (its size and digest, stored); the reference decodes it to the input
    (checked where the answer was made), so decoding our identical bytes checks both directions."""
    data = synth.zipf_text(1500, seed=8).tobytes()
    rc, got, _, _ = encode_file(L, tmp_path, data, 1 << 20, 2, "ref")
    assert rc == 0
    refs.check_answer("cli/zipf1500_seed8_b1", [len(got), refs.digest(got)])
    rc, back, _, _ = decode_bytes(L, tmp_path, got, 2, name="ref")
    assert rc == 0 and back == data


def test_error_paths_wind_the_pipeline_down(L, tmp_path, four_blocks):
    data, want = four_blocks
    E = bzip3_b200
    rc, _, _, _ = decode_bytes(L, tmp_path, b"BZ3v2" + want[5:], 3)
    assert rc == -21                                     # BZ3_B200_ERR_SIGNATURE
    rc, _, _, _ = decode_bytes(L, tmp_path, want[:7], 3)
    assert rc == -21
    rc, _, _, _ = decode_bytes(L, tmp_path, b"BZ3v1" + struct.pack("<i", 1000) + want[9:], 3)
    assert rc == -24                                     # BZ3_B200_ERR_BLOCK_SIZE
    # the file ends inside the third block: the two blocks before it are written, then TRUNCATED
    first = 9
    sizes = []
    at = first
    while at < len(want):
        c, o = struct.unpack_from("<ii", want, at)
        sizes.append((at, c, o))
        at += 8 + c
    cut = sizes[2][0] + 8 + sizes[2][1] // 2
    rc, back, _, _ = decode_bytes(L, tmp_path, want[:cut], 2)
    assert rc == -23 and back == data[:2 * BS]
    rc, back, _, _ = decode_bytes(L, tmp_path, want[:sizes[1][0] + 5], 4)   # ends inside a block header
    assert rc == -23 and back == data[:BS]
    # inconsistent headers (:265): original size beyond bz3_bound(block size), and a negative coded size
    bad = bytearray(want)
    struct.pack_into("<i", bad, sizes[1][0] + 4, bzip3_b200.bound(BS) + 1)
    rc, back, _, _ = decode_bytes(L, tmp_path, bytes(bad), 3)
    assert rc == -22 and back == data[:BS]
    bad = bytearray(want)
    struct.pack_into("<i", bad, sizes[0][0], -5)
    rc, back, _, _ = decode_bytes(L, tmp_path, bytes(bad), 3)
    assert rc == -22 and back == b""
    # a damaged payload: the block's own error comes back, the blocks before it are out, later ones are not
    bad = bytearray(want)
    bad[sizes[1][0] + 8 + sizes[1][1] // 2] ^= 0x41
    blk = bytes(bad[sizes[1][0] + 8: sizes[1][0] + 8 + sizes[1][1]])
    expect = refs.oracle_decode_block(blk, sizes[1][2], BS, err_init=55)
    assert expect[1] == -1
    rc, back, _, _ = decode_bytes(L, tmp_path, bytes(bad), 4)
    assert rc == expect[2] and back == data[:BS]
    rc, _, _, _ = decode_bytes(L, tmp_path, bytes(bad), 1, test_only=True)
    assert rc == expect[2]
    # encode: block size out of range, unwritable output
    assert L.bz3_b200_encode_fd(0, 1, 1000, 2, None, None) == -24
    src = tmp_path / "e.bin"
    src.write_bytes(data)
    fi = os.open(src, os.O_RDONLY)
    ro = os.open(src, os.O_RDONLY)   # a read-only descriptor as the output
    try:
        assert L.bz3_b200_encode_fd(fi, ro, BS, 2, None, None) == -20   # BZ3_B200_ERR_IO
    finally:
        os.close(fi)
        os.close(ro)


def test_command_line_tool(L, tmp_path):
    """bzip3_b200/bz3b200 (csrc/cli_main.cpp) on the emulator build: same bytes as the reference tool, -d / -t, exit codes."""
    cli = os.path.join(refs.ROOT, "bzip3_b200", "bz3b200")
    if not (os.path.exists(cli) and os.access(cli, os.X_OK)):
        pytest.skip("bzip3_b200/bz3b200 not built")
    env = dict(os.environ, BZ3_B200_LIB=build_emulated_library())
    data = synth.zipf_text(1800, seed=12).tobytes()
    src, packed, back = tmp_path / "a.txt", tmp_path / "a.bz3", tmp_path / "a.out"
    src.write_bytes(data)
    r = subprocess.run([cli, "-e", "-b", "1", "-j", "2", "-v", str(src), str(packed)], env=env, capture_output=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert b"MiB/s" in r.stderr
    assert packed.read_bytes() == container(data, 1 << 20)
    refs.check_answer("cli/zipf1800_seed12_b1", [len(packed.read_bytes()), refs.digest(packed.read_bytes())])
    assert subprocess.run([cli, "-e", str(src), str(packed)], env=env, capture_output=True).returncode == 1   # exists, no -f
    assert subprocess.run([cli, "-t", str(packed)], env=env, capture_output=True, timeout=300).returncode == 0
    r = subprocess.run([cli, "-d", str(packed), str(back)], env=env, capture_output=True, timeout=300)
    assert r.returncode == 0 and back.read_bytes() == data
    r = subprocess.run([cli, "-d", "-c"], input=packed.read_bytes(), env=env, capture_output=True, timeout=300)   # stdin -> stdout
    assert r.returncode == 0 and r.stdout == data
    blob = bytearray(packed.read_bytes())
    blob[len(blob) // 2] ^= 0x10
    r = subprocess.run([cli, "-t"], input=bytes(blob), env=env, capture_output=True, timeout=300)
    assert r.returncode == 1 and b"Failed to decode" in r.stderr
    r = subprocess.run([cli, "-d"], input=b"not a bz3 file", env=env, capture_output=True, timeout=300)
    assert r.returncode == 1 and b"invalid signature" in r.stderr


def test_gpu_many_blocks_check_runs_on_the_emulator(L):
    """The body of the GPU test of many blocks in flight (tests/test_gpu_stream.py), at emulator size."""
    from tests.test_gpu_stream import many_blocks_check
    many_blocks_check(L, BS, 4, 1300)


def test_dealing_workers_over_devices(L, tmp_path, four_blocks):
    """bz3_b200_*_fd2 with devices = 0 (all visible: one on the emulator) and more devices than exist."""
    data, want = four_blocks
    src, dst = tmp_path / "d.bin", tmp_path / "d.bz3"
    src.write_bytes(data)
    for devices in (5,):   # more devices than exist (one on the emulator); 0 = all visible is the GPU test's case
        fi, fo = os.open(src, os.O_RDONLY), os.open(dst, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
        try:
            assert L.bz3_b200_encode_fd2(fi, fo, BS, 3, devices, None, None) == 0
        finally:
            os.close(fi)
            os.close(fo)
        assert dst.read_bytes() == want


def reference_loop_model(blob, bs):
    """The decode loop of the reference tool (src/main.c:186-203, :257-278) restated around the oracle's block decoder:
    returns (code, output) with the codes of include/bz3_b200.h for what the tool reports as text."""
    if len(blob) < 9 or blob[:5] != b"BZ3v1":
        return -21, b""
    block_size = struct.unpack_from("<i", blob, 5)[0]
    if block_size < 65 * 1024 or block_size > 511 * 1024 * 1024:
        return -24, b""
    cap = bzip3_b200.bound(block_size)
    out = bytearray()
    at = 9
    while at < len(blob):
        if len(blob) - at < 8:
            return -23, bytes(out)
        new_size, old_size = struct.unpack_from("<ii", blob, at)
        if old_size < 0 or new_size < 0 or old_size > cap or new_size > cap:
            return -22, bytes(out)
        if len(blob) - at - 8 < new_size:
            return -23, bytes(out)
        blk = blob[at + 8: at + 8 + new_size]
        dec, r, err = refs.oracle_decode_block(blk, old_size, block_size, buffer_size=cap, compressed_size=new_size, err_init=55)
        if r == -1:
            return (err if err != 55 else -7), bytes(out)
        out += dec[:old_size] if len(dec) >= old_size else dec + bytes(old_size - len(dec))
        at += 8 + new_size
    return 0, bytes(out)


def test_mutated_containers_follow_the_reference_loop(L, tmp_path):
    """Random damage to a three-block container: same verdict and same bytes out as the reference tool's loop (modelled
    above around the oracle), whatever gets hit -- signature, block size, block headers, payload, the end of the file."""
    data, blobs = mutated_containers()
    assert reference_loop_model(container(data, BS), BS) == (0, data)
    pins = refs.reference_answer("mutated_containers")
    assert len(pins) == len(blobs)
    for trial, ((kind, blob), pin) in enumerate(zip(blobs, pins)):
        want = reference_loop_model(blob, BS)
        # the model itself is pinned on the reference binary: exit status and bytes written
        assert [want[0] == 0, refs.digest(want[1])] == pin, (trial, kind, want[0])
        rc, back, _, _ = decode_bytes(L, tmp_path, blob, 1 + trial % 3, name="m%d" % trial)
        assert rc == want[0], (trial, kind, rc, want[0])
        assert back == want[1], (trial, kind, len(back), len(want[1]))


def mutated_containers():
    """(data, [(kind, damaged container)]): 21 random kinds of damage to the container of three blocks of `data`."""
    data = squeezable(2 * BS + 3000, seed=9)
    good = container(data, BS)
    rng = np.random.default_rng(2026)
    offsets = [9]
    while offsets[-1] < len(good):
        offsets.append(offsets[-1] + 8 + struct.unpack_from("<i", good, offsets[-1])[0])
    blobs = []
    for trial in range(21):
        blob = bytearray(good)
        kind = trial % 7
        if kind == 0:      # a bit anywhere in a payload
            k = int(rng.integers(0, len(offsets) - 1))
            blob[int(rng.integers(offsets[k] + 8, offsets[k + 1]))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1:    # a byte of a block header
            k = int(rng.integers(0, len(offsets) - 1))
            blob[offsets[k] + int(rng.integers(0, 8))] ^= int(rng.integers(1, 256))
        elif kind == 2:    # cut anywhere
            blob = blob[: int(rng.integers(0, len(blob)))]
        elif kind == 3:    # the first bytes of a block's own header (checksum / BWT index / model)
            k = int(rng.integers(0, len(offsets) - 1))
            blob[offsets[k] + 8 + int(rng.integers(0, 9))] ^= int(rng.integers(1, 256))
        elif kind == 4:    # container header
            blob[int(rng.integers(0, 9))] ^= int(rng.integers(1, 256))
        elif kind == 5:    # original size of a block lowered / raised a little
            k = int(rng.integers(0, len(offsets) - 1))
            o = struct.unpack_from("<i", blob, offsets[k] + 4)[0]
            struct.pack_into("<i", blob, offsets[k] + 4, max(0, o + int(rng.integers(-70, 70))))
        else:              # trailing garbage
            blob += bytes(rng.integers(0, 256, int(rng.integers(1, 12)), dtype=np.uint8))
        blobs.append((kind, bytes(blob)))
    return data, blobs


def test_workers_without_a_state_borrow_one(tmp_path):
    """Device memory for two states, six workers: the four whose bz3_new() fails code their blocks on a state of the other
    two (one block at a time per state) instead of ending the stream with BZ3_ERR_INIT after part of the output is written.
    A device with no room for any state still reports BZ3_ERR_INIT.  Runs in a subprocess: the memory cap of the emulated
    device (BZ_EMU_MALLOC_TOTAL) is read from the environment."""
    import sys
    so = build_emulated_library()
    data = squeezable(11 * BS + 1234, seed=91)
    (tmp_path / "in.bin").write_bytes(data)
    (tmp_path / "want.bz3").write_bytes(container(data, BS))
    script = (
        "import ctypes as C, os, sys\n"
        "sys.path.insert(0, %r)\n"
        "import bzip3_b200\n"
        "L = bzip3_b200.lib()\n"
        "d = %r\n"
        "fi = os.open(d + '/in.bin', os.O_RDONLY); fo = os.open(d + '/out.bz3', os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)\n"
        "nin, nout = C.c_uint64(0), C.c_uint64(0)\n"
        "rc = L.bz3_b200_encode_fd(fi, fo, %d, 6, C.byref(nin), C.byref(nout)); os.close(fi); os.close(fo)\n"
        "print('ENC', rc, open(d + '/out.bz3', 'rb').read() == open(d + '/want.bz3', 'rb').read())\n"
        "fi = os.open(d + '/want.bz3', os.O_RDONLY); fo = os.open(d + '/back.bin', os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)\n"
        "rc = L.bz3_b200_decode_fd(fi, fo, 6, C.byref(nin), C.byref(nout)); os.close(fi); os.close(fo)\n"
        "print('DEC', rc, open(d + '/back.bin', 'rb').read() == open(d + '/in.bin', 'rb').read())\n" % (refs.ROOT, str(tmp_path), BS))
    own = 3.2 * bzip3_b200.bound(BS) + (1 << 20) + 8192        # what a state owns (test_emu_library)
    for total, want in ((int(2 * 52 * BS + 2.5 * own), ("ENC 0 True", "DEC 0 True")),      # two workspaces + two states
                        (int(0.5 * own), ("ENC %d False" % bzip3_b200.BZ3_ERR_INIT, "DEC %d False" % bzip3_b200.BZ3_ERR_INIT))):
        env = dict(os.environ, BZ3_B200_LIB=so, BZ_EMU_MALLOC_TOTAL=str(total))
        out = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=900)
        assert all(w in out.stdout for w in want), (total, out.stdout, out.stderr[-2000:])
