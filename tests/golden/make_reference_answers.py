"""Writes tests/golden/reference_answers.json: what the unmodified reference computes for the inputs of every test that
compares with it, as return values and digests of the bytes written (refs.digest).  The tests read only this file.

Needs the reference built into oracle/_ref (`make -C oracle ref REF=<checkout of the reference>`).  Takes a few
minutes, most of it the 256 MiB and 511 MiB blocks.  Usage, from the repository root:

    python tests/golden/make_reference_answers.py
"""
import ctypes as C
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from bzip3_b200 import synth  # noqa: E402
from tests import refs, test_abi, test_emu_kernels, test_emu_library, test_emu_stream  # noqa: E402
from tests import test_gpu_large, test_gpu_stream  # noqa: E402
from tests import test_oracle as T  # noqa: E402

L = refs.ref()
R = refs.ref_stages()


def ref_bwt(src, dst, n):
    A = np.zeros(n + 256, np.int32)
    return R.ref_bwt(src, dst, A.ctypes.data_as(refs.i32p), n)


def ref_unbwt(src, dst, n, idx):
    A = np.zeros(n + 256, np.int32)
    return R.ref_unbwt(src, dst, A.ctypes.data_as(refs.i32p), n, idx)


# the reference's stage and block functions with the calling convention of test_oracle.ORACLE_STAGES / ORACLE_BLOCKS
STAGES = SimpleNamespace(crc=R.ref_crc32, mrle_encode=R.ref_mrlec, mrle_decode=R.ref_mrled,
                         lzp_encode=lambda src, n, dst, lut: R.ref_lzp_compress(src, dst, n, lut),
                         lzp_decode=lambda src, insize, dst, cap, lut: R.ref_lzp_decompress(src, dst, insize, cap, lut),
                         bwt=ref_bwt, unbwt=ref_unbwt, cm_encode=R.ref_cm_encode, cm_decode=R.ref_cm_decode)
BLOCKS = SimpleNamespace(
    encode=lambda data, bs: refs.api_encode_block(L, data, bs),
    decode=lambda enc, osz, bs, buffer_size=None, compressed_size=None: refs.api_decode_block(
        L, enc, osz, bs, buffer_size=buffer_size, compressed_size=compressed_size))


def block(data, bs):
    """[return value, last error, digest] of bz3_encode_block; the reference must decode its block to the input."""
    enc, r, e = BLOCKS.encode(bytes(data), bs)
    assert BLOCKS.decode(enc, len(data), bs)[0] == bytes(data)
    return [r, e, refs.digest(enc)]


def frame(block_size, data):
    """[size, digest] of bz3_compress; the reference must decompress its frame to the input."""
    data = np.frombuffer(bytes(data), np.uint8)
    out = np.zeros(refs.bound(len(data)) + 64, np.uint8)
    osz = C.c_size_t(len(out))
    assert L.bz3_compress(block_size, refs.ptr(data), refs.ptr(out), len(data), C.byref(osz)) == 0
    back = np.zeros(len(data) + 64, np.uint8)
    bsz = C.c_size_t(len(back))
    assert L.bz3_decompress(refs.ptr(out), refs.ptr(back), osz.value, C.byref(bsz)) == 0
    assert bytes(back[:bsz.value]) == data.tobytes()
    return [osz.value, refs.digest(out[:osz.value])]


def cli(data, *args):
    """[size, digest] of the file `bzip3 -e ARGS` writes; the reference tool must decode it to the input."""
    enc = subprocess.run([refs.REF_CLI, "-e", *args], input=data, capture_output=True, check=True, timeout=900).stdout
    dec = subprocess.run([refs.REF_CLI, "-d"], input=enc, capture_output=True, check=True, timeout=900).stdout
    assert dec == data
    return [len(enc), refs.digest(enc)]


def answers():
    a = {}
    for name, data in T.CASES:
        a[f"stage_crc/{name}"] = T.crc_answer(STAGES, data)
        a[f"stage_mrle/{name}"] = T.mrle_answer(STAGES, data)
        a[f"stage_lzp/{name}"] = T.lzp_answer(STAGES, data)
        a[f"stage_bwt/{name}"] = T.bwt_answer(STAGES, data)
        a[f"stage_cm/{name}"] = T.cm_answer(STAGES, data)
        a[f"block/{name}"] = T.block_answer(BLOCKS, data)
    a["block_too_big"] = list(BLOCKS.encode(bytes(70000), 65 * 1024)[1:])
    for name in T.HOSTILE:
        a[f"hostile/{name}"] = T.hostile_answer(BLOCKS, name)
    a["medium_corpora"] = T.medium_answer(BLOCKS, T.medium_corpora())
    a["min_memory_needed"] = [L.bz3_min_memory_needed(bs) for bs in test_abi.MIN_MEMORY_BLOCK_SIZES]

    n, payloads = test_emu_kernels.exhausted_payloads()
    pins = []
    for buf, insize in payloads:
        pin = np.zeros(n + 8, np.uint8)
        R.ref_cm_decode(refs.ptr(buf.copy()), insize, refs.ptr(pin), n)
        pins.append(refs.digest(pin[:n]))
    a["cm_exhausted"] = pins

    _, blobs = test_emu_stream.mutated_containers()
    pins = []
    for _, blob in blobs:
        r = subprocess.run([refs.REF_CLI, "-d"], input=blob, capture_output=True, timeout=120)
        pins.append([r.returncode == 0, refs.digest(r.stdout)])
    a["mutated_containers"] = pins

    a["frame/zipf2200_seed9"] = frame(test_emu_library.BS, synth.zipf_text(2200, seed=9))
    a["frame/zipf300k_seed11_b128k"] = frame(1 << 17, synth.zipf_text(300_000, seed=11))
    a["cross/zipf500k_seed21_b1m"] = block(synth.zipf_text(500_000, seed=21), 1 << 20)
    a["cli/zipf1500_seed8_b1"] = cli(synth.zipf_text(1500, seed=8).tobytes(), "-b", "1")
    a["cli/zipf1800_seed12_b1"] = cli(synth.zipf_text(1800, seed=12).tobytes(), "-b", "1")
    a["cli/stream_corpus_b1"] = cli(test_gpu_stream.corpus_data(), "-b", "1", "-j", "4")
    # the input of tests/test_gpu_multi.py::test_tools_over_all_gpus
    a["cli/source_5mib_b1"] = cli(synth.source_corpus(5 * (1 << 20) + 12345, seed=61).tobytes(), "-b", "1", "-j", "4")
    a["large/batch_16mib"] = [block(d, 16 << 20)[0::2] for d in test_gpu_large.batch_16mib_data()]
    for key, make in test_gpu_large.BLOCKS.items():
        data = make()
        a[key] = block(data, len(data))
        print(key, a[key], flush=True)
    return a


def main():
    a = answers()
    with open(refs.ANSWERS, "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in sorted(a.items())) + "\n}\n")
    print(f"wrote {len(a)} answers to {os.path.relpath(refs.ANSWERS, ROOT)}")


if __name__ == "__main__":
    main()
