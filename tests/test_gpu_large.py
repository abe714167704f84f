"""Large blocks on the GPU against the reference: the encoded block must equal the reference's bz3_encode_block output
byte for byte (its size and digest, tests/golden/reference_answers.json) and decode, up to the metric's block size
(256 MiB, BASELINE.json configs[2]) and the format's maximum (511 MiB, configs[4]; src/libbz3.c:536); plus the batch API
at the benchmark's block size.  The reference decodes each of its blocks to the input where the answers were made, so
a block equal to the reference's decodes there too."""
import struct

import numpy as np
import pytest

import bzip3_b200
from bzip3_b200 import synth
from tests import refs

pytestmark = pytest.mark.gpu

# the single blocks compared with the reference's: answer key -> a function making their bytes
BLOCKS = {
    "large/source_64mib": lambda: synth.source_corpus(64 << 20, seed=1234 + 64),
    "large/mixed_32mib": lambda: synth.mixed(32 << 20, seed=1234 + 32, segment=4 << 20),
    "large/source_256mib": lambda: synth.source_corpus(256 << 20, seed=synth.SEED_SOURCE),
    "large/log_511mib": lambda: synth.log_stream(511 << 20, seed=synth.SEED_LOG),
}


def roundtrip(key):
    data = BLOCKS[key]()
    n = len(data)
    with bzip3_b200.Bz3State(n) as s:
        enc, r = s.encode_block(data.tobytes())
        assert r > 0 and s.last_error == 0
        crc, idx, model = struct.unpack("<IiB", enc[:9])
        assert crc == refs.oracle().orc_crc32(1, refs.ptr(data), n)
        assert 1 <= idx <= n
        refs.check_answer(key, [r, s.last_error, refs.digest(enc)])
        dec, r2 = s.decode_block(enc, n)
        assert r2 == n and s.last_error == 0 and dec == data.tobytes()


def test_roundtrip_64mib_source_block():
    roundtrip("large/source_64mib")


def test_roundtrip_32mib_mixed_block_with_incompressible_segments():
    roundtrip("large/mixed_32mib")


def test_batch_of_16mib_blocks_matches_reference():
    bs = 16 << 20
    datas = batch_16mib_data()
    states = [bzip3_b200.Bz3State(bs) for _ in datas]
    try:
        bufs = []
        for d in datas:
            b = np.zeros(bzip3_b200.bound(bs) + 64, np.uint8)
            b[:len(d)] = np.frombuffer(d, np.uint8)
            bufs.append(b)
        sizes = bzip3_b200.encode_blocks(states, bufs, [len(d) for d in datas])
        assert all(s.last_error == 0 for s in states)
        refs.check_answer("large/batch_16mib", [[sz, refs.digest(b[:sz])] for b, sz in zip(bufs, sizes)])
        bzip3_b200.decode_blocks(states, bufs, [len(b) for b in bufs], sizes, [len(d) for d in datas])
        for d, b, s in zip(datas, bufs, states):
            assert s.last_error == 0 and bytes(b[:len(d)]) == d
    finally:
        for s in states:
            s.close()


def batch_16mib_data():
    bs = 16 << 20
    return [synth.zipf_text(bs, seed=77).tobytes(), synth.log_stream(bs // 2, seed=78).tobytes()]


def test_many_blocks_of_mixed_sizes_at_once():
    """40 states with different block sizes coded by 40 host threads at once, twice: sorts with different pass counts
    (8 for the first round of a suffix sort, 2 * ceil(log2(n + 1)) / 8 afterwards, 3 for LZP, 1 for the inverse BWT) overlap
    in time, so every per-function launch attribute must be the same for all of them.  (A histogram kernel whose shared
    memory limit followed the launching thread's pass count failed here with "too many resources requested for launch".)"""
    rng = np.random.default_rng(4040)
    sizes = [int(x) for x in rng.integers(70 << 10, 3 << 20, 40)]
    gens = [synth.zipf_text, synth.source_corpus, synth.log_stream]
    datas = [gens[i % 3](n, seed=500 + i).tobytes()[:n] for i, n in enumerate(sizes)]
    states = [bzip3_b200.Bz3State(max(len(d), 65 << 10)) for d in datas]
    try:
        for rep in range(2):
            bufs = []
            for d in datas:
                b = np.zeros(bzip3_b200.bound(len(d)) + 64, np.uint8)
                b[:len(d)] = np.frombuffer(d, np.uint8)
                bufs.append(b)
            enc = bzip3_b200.encode_blocks(states, bufs, [len(d) for d in datas])
            assert all(s.last_error == 0 for s in states), [s.last_error for s in states]
            assert all(e > 0 for e in enc), enc
            if rep == 0:
                for i in (0, 1, 2, 17, 39):
                    want, r, _ = refs.oracle_encode_block(datas[i], max(len(datas[i]), 65 << 10))
                    assert r == enc[i] and want == bytes(bufs[i][:enc[i]]), i
            bzip3_b200.decode_blocks(states, bufs, [len(b) for b in bufs], enc, [len(d) for d in datas])
            for d, b, s in zip(datas, bufs, states):
                assert s.last_error == 0 and bytes(b[:len(d)]) == d
    finally:
        for s in states:
            s.close()


def _against_reference_big(key):
    """encode on the GPU, compare with the reference's block, decode"""
    data = BLOCKS[key]()
    n = len(data)
    L = bzip3_b200.lib()
    cap = refs.bound(n) + 64
    gbuf = np.zeros(cap, np.uint8)
    gbuf[:n] = data
    with bzip3_b200.Bz3State(n) as s:
        r = L.bz3_encode_block(s.handle, refs.ptr(gbuf), n)
        assert r > 0 and s.last_error == 0, (r, s.last_error)
        refs.check_answer(key, [r, s.last_error, refs.digest(gbuf[:r])])
        r2 = L.bz3_decode_block(s.handle, refs.ptr(gbuf), cap, r, n)
        assert r2 == n and s.last_error == 0, (r2, s.last_error)
        assert np.array_equal(gbuf[:n], data), "GPU decode of the block differs from the input"


def test_256mib_block_equals_the_reference():
    """the metric's block size: one 256 MiB block of the synthetic source corpus (BASELINE.json configs[2])"""
    _against_reference_big("large/source_256mib")


def test_511mib_block_equals_the_reference():
    """the largest block the format allows (src/libbz3.c:536): 511 MiB of the synthetic log stream (configs[4])"""
    _against_reference_big("large/log_511mib")
