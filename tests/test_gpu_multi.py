"""Several GPUs from ONE process through the reference ABI (SURVEY.md 8b "GPU mapping", 8e): bz3_new() deals states over
the visible devices (bz3_b200_set_devices / BZ3_B200_DEVICES), so the reference's batch calls run block i on GPU i mod N;
the reference's own front end (src/main.c, -j N) and the bz3b200 tool (-g N) do the same.  Needs at least two GPUs
(`python -m pytest tests/test_gpu_multi.py -m gpu` on a machine with two or more); skipped on a one-GPU machine."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import bzip3_b200
from bzip3_b200 import synth
from tests import refs

pytestmark = pytest.mark.gpu
BS = 1 << 20


def ngpus():
    try:
        return bzip3_b200.lib().bz3_b200_device_count()
    except Exception:
        return 0


needs2 = pytest.mark.skipif(ngpus() < 2, reason="needs at least two GPUs")


@needs2
def test_batch_api_deals_blocks_over_the_gpus():
    L = bzip3_b200.lib()
    g = L.bz3_b200_set_devices(0)   # all visible
    assert g == ngpus()
    try:
        nblk = 2 * g + 1
        datas = [synth.zipf_text(BS - 1000 * k, seed=50 + k).tobytes() for k in range(nblk)]
        states = [bzip3_b200.Bz3State(BS) for _ in datas]
        try:
            devs = [L.bz3_b200_state_device(s.handle) for s in states]
            assert sorted(set(devs)) == list(range(g)), devs            # every GPU got states ...
            assert all(devs[k + g] == devs[k] for k in range(nblk - g))   # ... round-robin
            bufs = []
            for d in datas:
                b = np.zeros(bzip3_b200.bound(BS) + 64, np.uint8)
                b[:len(d)] = np.frombuffer(d, np.uint8)
                bufs.append(b)
            sizes = bzip3_b200.encode_blocks(states, bufs, [len(d) for d in datas])
            assert all(s.last_error == 0 for s in states)
            for d, b, sz in zip(datas, bufs, sizes):
                want = refs.oracle_encode_block(d, BS)
                assert sz == want[1] and bytes(b[:sz]) == want[0]
            bzip3_b200.decode_blocks(states, bufs, [len(b) for b in bufs], sizes, [len(d) for d in datas])
            for d, b, s in zip(datas, bufs, states):
                assert s.last_error == 0 and bytes(b[:len(d)]) == d
        finally:
            for s in states:
                s.close()
    finally:
        L.bz3_b200_set_devices(1)


@needs2
def test_tools_over_all_gpus(tmp_path):
    """the reference's unmodified front end on the library with BZ3_B200_DEVICES=all, and bz3b200 -g 0"""
    data = synth.source_corpus(5 * BS + 12345, seed=61).tobytes()
    src = tmp_path / "in.bin"
    src.write_bytes(data)
    outs = {}
    cli_b200 = os.path.join(refs.ROOT, "oracle", "_ref", "bzip3_cli_on_b200")
    tool = os.path.join(refs.ROOT, "bzip3_b200", "bz3b200")
    cmds = {"bz3b200": [tool, "-e", "-b", "1", "-g", "0", "-c", str(src)]}
    if os.path.exists(cli_b200):
        cmds["ref_cli_on_lib"] = [cli_b200, "-e", "-b", "1", "-j", "4"]
    for name, cmd in cmds.items():
        env = dict(os.environ)
        if name == "ref_cli_on_lib":   # the reference's front end knows nothing about GPUs: the library deals its states
            env["BZ3_B200_DEVICES"] = "all"
        with open(src, "rb") as fi:
            r = subprocess.run(cmd, stdin=fi, capture_output=True, env=env, timeout=900)
        assert r.returncode == 0, (name, r.stderr[-500:])
        outs[name] = r.stdout
    first = next(iter(outs.values()))
    assert all(v == first for v in outs.values()), {k: len(v) for k, v in outs.items()}
    refs.check_answer("cli/source_5mib_b1", [len(first), refs.digest(first)])   # what `bzip3 -e -b 1 -j 4` writes
    r = subprocess.run([tool, "-d", "-g", "0", "-c"], input=first, capture_output=True, timeout=900)
    assert r.returncode == 0 and r.stdout == data
