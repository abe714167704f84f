#!/usr/bin/env python
"""bench.py -- round-trip (encode + decode) throughput of the bzip3 block codec on B200.

One "step" = bz3_encode_blocks + bz3_decode_blocks over every block of the rank's workload (all blocks in flight at once,
one stream per block), i.e. one full round trip of the rank's data through the reference ABI on pinned HOST buffers.

  e2e        MiB/s of uncompressed data through the K timed steps above (H2D + D2H inside the timed region; for N > 1 also
             the NCCL gather of the compressed blocks to rank 0, bzip3_b200/sharding.py).  `ms_per_step` is this loop's.
  value      the same round trip with the inputs already resident in HBM (bz3_b200_encode_resident_many /
             bz3_b200_decode_resident_many), a side loop of W warm-up + K timed steps: the two differ by the PCIe copies
             only (< 0.1 %).
  headline_b256   BASELINE.json's metric configuration (1 GiB synthetic source corpus, -b 256, 4 blocks of 256 MiB per
             GPU): 1 warm-up + 1 timed e2e step, block 0 compared with the reference encoder, the reference's pthread
             path timed on the same bytes.  Skipped with --no-headline or when the run is already late.
  roofline   dominant kernel (by device time) vs the measured HBM peak, plus the suffix-sort radix passes.
  cpu_baseline / --impl reference : the unmodified reference (oracle/_ref/libbz3_ref.so, built from /root/reference by
             oracle/Makefile) on the host cores: bz3_encode_blocks / bz3_decode_blocks in batches of min(cores, 64)
             pthreads like src/main.c:352-378, on the bytes of the WHOLE job (all N ranks' workloads).

Launch: python bench.py [--gpus N --steps K --warmup W]  or, for N>1,
        python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...
"""
from __future__ import annotations

import os as _os

# One CUDA stream per block: give every stream its own hardware queue, otherwise a copy queued behind one
# block's seconds-long coder kernel falsely serialises the other blocks' short kernels (must be set before
# the CUDA context exists).
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
# One stage workspace per block of a 4-block batch (library default: 2).  On match-dense data the LZP stage holds a
# workspace for seconds (3 s per 256 MiB block of the source corpus), so with two of them the third and fourth block of
# the metric's configuration start their coder 3 s late.  Same knob a caller of the library has (INTEGRATION.md).
_os.environ.setdefault("BZ3_B200_ARENAS", "4")

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bzip3_b200 import synth  # noqa: E402

MIB = float(1 << 20)
T_START = time.time()

WORKLOADS = {
    # BASELINE.json configs[1]: "enwik8-style 100 MB synthetic Zipf text, -b 16, 1 GPU"
    "zipf100m_b16": dict(gen="zipf_text", nbytes=100_000_000, block=16 << 20, seed=synth.SEED_ZIPF_TEXT,
                         desc="100 MB synthetic Zipf(1.1) text, -b 16 (6 blocks: 5 x 16 MiB + 16 113 920 B)"),
    # BASELINE.json configs[2] / the metric's configuration: "1 GiB synthetic source-code corpus, -b 256"
    "src1g_b256": dict(gen="source_corpus", nbytes=1 << 30, block=256 << 20, seed=synth.SEED_SOURCE,
                       desc="1 GiB synthetic source corpus, -b 256 (4 blocks of 256 MiB)"),
    # BASELINE.json configs[3] per GPU: "8 GiB mixed text+binary, -b 256, 8 GPUs block-sharded" = 1 GiB, 4 blocks per GPU
    "mixed1g_b256": dict(gen="mixed", nbytes=1 << 30, block=256 << 20, seed=synth.SEED_MIXED,
                         desc="1 GiB per GPU of the mixed text+binary stream (64 MiB segments), -b 256 (4 blocks per GPU)"),
    # BASELINE.json configs[4] per GPU, scaled to what one step can afford: log stream, -b 511
    "log2g_b511": dict(gen="log_stream", nbytes=4 * (511 << 20), block=511 << 20, seed=synth.SEED_LOG,
                       desc="2044 MiB per GPU of the synthetic log stream, -b 511 (4 blocks of 511 MiB per GPU)"),
    "src256m_b64": dict(gen="source_corpus", nbytes=256 << 20, block=64 << 20, seed=synth.SEED_SOURCE,
                        desc="256 MiB synthetic source corpus, -b 64 (4 blocks)"),
    # not a BASELINE config: many blocks per GPU, to measure what blocks in flight buy (tools/inflight_curve.py)
    "zipf2g_b16": dict(gen="zipf_text", nbytes=2 << 30, block=16 << 20, seed=synth.SEED_ZIPF_TEXT,
                       desc="2 GiB synthetic Zipf(1.1) text, -b 16 (128 blocks in flight per GPU)"),
    "zipf8m_b1": dict(gen="zipf_text", nbytes=8 << 20, block=1 << 20, seed=synth.SEED_ZIPF_TEXT,
                      desc="8 MiB synthetic Zipf text, -b 1 (8 blocks) -- quick self-test"),
}
HEADLINE = "src1g_b256"


def load_workload(name: str, rank: int):
    """The rank's share of the job: its own synthetic stream (seed + 1000 * rank), cut into blocks."""
    w = WORKLOADS[name]
    seed = w["seed"] + 1000 * rank
    cache_dir = os.environ.get("BZ3_B200_CACHE", "/tmp/bz3_b200_cache")
    path = os.path.join(cache_dir, f"{name}_{seed:x}.bin")
    data = None
    if os.path.exists(path) and os.path.getsize(path) == w["nbytes"]:
        data = np.fromfile(path, dtype=np.uint8)
    if data is None:
        data = getattr(synth, w["gen"])(w["nbytes"], seed=seed)
        try:
            os.makedirs(cache_dir, exist_ok=True)
            data.tofile(path)
        except OSError:
            pass
    bs = w["block"]
    blocks = [data[i:i + bs] for i in range(0, len(data), bs)]
    return blocks, bs, w


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx = max(mx, float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------- reference arm
def reference_lib():
    from tests import refs
    if refs.have_ref():
        return refs.ref(), "reference"
    return None, "port"


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def reference_jobs():
    """-j of the reference tool on this host: its worker count is capped at 64 (src/main.c:213)."""
    return max(1, min(host_threads(), 64))


def reference_roundtrip(blocks, bs, jobs, check=True):
    """One round trip with the reference's own batch API (pthread per block, batches of `jobs` like src/main.c:352-378).
    Returns (seconds_encode, seconds_decode, kind, threads_used)."""
    from tests import refs
    R, kind = reference_lib()
    cap = refs.bound(bs) + 64
    if R is None:  # oracle port, single thread
        te = td = 0.0
        for b in blocks:
            buf = np.zeros(cap, np.uint8)
            buf[:len(b)] = b
            err = C.c_int8(0)
            t0 = time.perf_counter()
            r = refs.oracle().orc_encode_block(bs, refs.ptr(buf), len(b), C.byref(err))
            t1 = time.perf_counter()
            refs.oracle().orc_decode_block(bs, refs.ptr(buf), cap, r, len(b), C.byref(err))
            t2 = time.perf_counter()
            te += t1 - t0
            td += t2 - t1
            assert bytes(buf[:len(b)]) == b.tobytes()
        return te, td, kind, 1
    used = min(jobs, len(blocks))
    states = [R.bz3_new(bs) for _ in range(used)]
    assert all(states), "the reference's bz3_new failed (host memory?)"
    bufs = [np.zeros(cap, np.uint8) for _ in states]
    te = td = 0.0
    try:
        for a in range(0, len(blocks), used):
            grp = blocks[a:a + used]
            n = len(grp)
            for b, buf in zip(grp, bufs):
                buf[:len(b)] = b
            hs = (C.c_void_p * n)(*states[:n])
            bp = (refs.u8p * n)(*[refs.ptr(x) for x in bufs[:n]])
            sz = (C.c_int32 * n)(*[len(b) for b in grp])
            t0 = time.perf_counter()
            R.bz3_encode_blocks(hs, bp, sz, n)
            t1 = time.perf_counter()
            bsz = (C.c_size_t * n)(*[cap] * n)
            osz = (C.c_int32 * n)(*[len(b) for b in grp])
            R.bz3_decode_blocks(hs, bp, bsz, sz, osz, n)
            t2 = time.perf_counter()
            te += t1 - t0
            td += t2 - t1
            if check:
                for b, buf, st in zip(grp, bufs, states):
                    assert R.bz3_last_error(st) == 0 and bytes(buf[:len(b)]) == b.tobytes()
    finally:
        for st in states:
            R.bz3_free(st)
    return te, td, kind, used


def run_reference_arm(args, rank, world):
    """The reference's own CPU path on the bytes of the whole job: the workloads of ranks 0 .. N-1, coded by
    min(host cores, 64) pthreads in batches like `bzip3 -j` (src/main.c:213, 352-378).  Rank 0 alone runs it."""
    if rank != 0:
        return
    n_ranks = max(1, args.gpus)
    blocks, bs, w = [], 0, None
    for r in range(n_ranks):
        b, bs, w = load_workload(args.workload, r)
        blocks += b
    total = sum(len(b) for b in blocks)
    jobs = reference_jobs()
    times = []
    kind, used = "reference", 1
    for i in range(args.warmup + args.steps):
        te, td, kind, used = reference_roundtrip(blocks, bs, jobs, check=(i == 0))
        if i >= args.warmup:
            times.append((te, td))
    te = sum(t[0] for t in times) / len(times)
    td = sum(t[1] for t in times) / len(times)
    ms = (te + td) * 1e3
    val = total / MIB / (te + td)
    out = {
        "impl": "reference", "metric": "roundtrip_MiB_per_s", "value": round(val, 3), "unit": "MiB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": args.workload, "description": w["desc"], "block_size": bs, "blocks": len(blocks),
                   "bytes": total, "job": f"the workloads of {n_ranks} rank(s), i.e. the same bytes the {n_ranks}-GPU arm codes"},
        "encode_MiB_per_s": round(total / MIB / te, 3), "decode_MiB_per_s": round(total / MIB / td, 3),
        "cpu_baseline": {"value": round(val, 3), "unit": "MiB/s", "cores": used, "kind": kind,
                         "sample": f"every step = the whole job ({len(blocks)} blocks, {total} B): bz3_encode_blocks / "
                                   f"bz3_decode_blocks in batches of {used} pthreads (-j min(cores, 64) = {jobs}; host has "
                                   f"{host_threads()} usable cores; gcc -O2 build of the unmodified reference)"},
        "e2e": {"value": round(val, 3), "unit": "MiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(out)


# ------------------------------------------------------------------------------------------- B200 arm
DUMP_SAMPLE = 7_500_000   # float32 values per byte array written by --dump-outputs: 60 MB for the two, under 64 MB


def dump_outputs(path, comp_sizes, compressed, decoded):
    """--dump-outputs: what the last timed step handed back to its caller, as DIR/<name>.npy.  Bytes are stored as
    float32 (exact).  A byte array longer than DUMP_SAMPLE is replaced by its values at DUMP_SAMPLE sorted indices drawn
    from a fixed seed, so two builds that return arrays of the same length are sampled at the same places."""
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "compressed_sizes.npy"), np.asarray(comp_sizes, np.float64))
    for name, a in (("compressed_bytes", compressed), ("decoded_bytes", decoded)):
        if a.size > DUMP_SAMPLE:
            a = a[np.sort(np.random.default_rng(2026).integers(0, a.size, DUMP_SAMPLE))]
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float32))


class Job:
    """The rank's blocks, one bz3_state per block, pinned host buffers for the ABI path."""

    def __init__(self, name, rank, torch, L, bzip3_b200, refs):
        self.name, self.L, self.refs, self.torch = name, L, refs, torch
        self.blocks, self.bs, self.w = load_workload(name, rank)
        self.nb = len(self.blocks)
        self.total = sum(len(b) for b in self.blocks)
        self.states = [bzip3_b200.Bz3State(self.bs) for _ in self.blocks]
        self.hs = (C.c_void_p * self.nb)(*[s.handle for s in self.states])
        self.osz = (C.c_int32 * self.nb)(*[len(b) for b in self.blocks])
        self.cap = bzip3_b200.bound(self.bs) + 64
        self.pinned = [torch.empty(self.cap, dtype=torch.uint8, pin_memory=True) for _ in self.blocks]
        self.bp = (refs.u8p * self.nb)(*[C.cast(p.data_ptr(), refs.u8p) for p in self.pinned])
        self.bsz = (C.c_size_t * self.nb)(*[self.cap] * self.nb)
        self.comp = [0] * self.nb

    def stage_host(self):
        for p, b in zip(self.pinned, self.blocks):
            p[:len(b)] = self.torch.from_numpy(b)

    def encode_abi(self):
        csz = (C.c_int32 * self.nb)(*[len(b) for b in self.blocks])
        self.L.bz3_encode_blocks(self.hs, self.bp, csz, self.nb)
        self.comp = [int(c) for c in csz]
        assert all(s.last_error == 0 for s in self.states) and min(self.comp) > 0, self.comp
        return csz

    def decode_abi(self, csz):
        self.L.bz3_decode_blocks(self.hs, self.bp, self.bsz, csz, self.osz, self.nb)
        assert all(s.last_error == 0 for s in self.states)

    def check_block0_against_reference(self):
        """bit-exactness gate: block 0 as coded through the ABI equals the reference encoder's output (any size)."""
        R, kind = reference_lib()
        if R is None:
            return "no reference library"
        want = self.refs.api_encode_block(R, self.blocks[0].tobytes(), self.bs)[0]
        got = bytes(self.pinned[0][:self.comp[0]].numpy())
        assert want == got, "block 0 differs from the reference encoder"
        return "block 0 (%d B) identical to the reference's bz3_encode_block output" % len(self.blocks[0])

    def close(self):
        for s in self.states:
            s.close()


def run_b200_arm(args, rank, world, local_rank):
    import torch
    import bzip3_b200
    from bzip3_b200 import sharding
    from tests import refs

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the codec has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    L = bzip3_b200.lib()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def e2e_step(job, keep=None):
        """encode + (N > 1: ordered gather of the compressed blocks to rank 0) + decode through the ABI on host buffers;
        `keep` (a list) receives the compressed blocks, which the decode overwrites in place"""
        job.stage_host()
        flush.fill_(1)
        barrier()
        ev[0].record()
        csz = job.encode_abi()
        if keep is not None:
            keep.extend(p[:c].numpy().copy() for p, c in zip(job.pinned, job.comp))
        if dist:  # the path's only exchange (SURVEY.md 8e): sizes by all_gather, padded payloads gathered to rank 0
            mine = {rank + k * world: job.pinned[k][:c].numpy() for k, c in enumerate(job.comp)}
            sharding.gather_compressed(mine, job.nb * world, rank, world, dist)
        job.decode_abi(csz)
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1])

    def reduce_max(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    job = Job(args.workload, rank, torch, L, bzip3_b200, refs)
    nb, total = job.nb, job.total
    job_bytes = reduce_sum(total)

    def gated_roundtrip(j):
        """one untimed round trip through the ABI: block 0 against the reference encoder, every block restored"""
        j.stage_host()
        csz = j.encode_abi()
        verdict = j.check_block0_against_reference() if rank == 0 else None
        j.decode_abi(csz)
        for p, b in zip(j.pinned, j.blocks):
            assert bytes(p[:len(b)].numpy()) == b.tobytes(), "round trip mismatch"
        return verdict

    gate = gated_roundtrip(job)
    gate_comp = list(job.comp)

    # ---------------- device-resident side loop: W warm-up + K timed steps
    sizes = (C.c_int32 * nb)(*[len(b) for b in job.blocks])
    enc_sizes = (C.c_int32 * nb)()
    dec_res = (C.c_int32 * nb)()
    res_ms = []
    for i in range(args.warmup + args.steps):
        for s, b in zip(job.states, job.blocks):
            assert L.bz3_b200_upload(s.handle, refs.ptr(b), len(b)) == 0
        flush.fill_(1)
        barrier()
        ev[0].record()
        L.bz3_b200_encode_resident_many(job.hs, sizes, enc_sizes, nb)
        ev[1].record()
        L.bz3_b200_decode_resident_many(job.hs, enc_sizes, job.osz, dec_res, nb)
        ev[2].record()
        torch.cuda.synchronize()
        assert list(dec_res) == [len(b) for b in job.blocks], list(dec_res)
        if i >= args.warmup:
            res_ms.append((ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])))
    res_enc = reduce_max(sum(t[0] for t in res_ms) / len(res_ms))
    res_dec = reduce_max(sum(t[1] for t in res_ms) / len(res_ms))
    res_step = reduce_max(sum(t[0] + t[1] for t in res_ms) / len(res_ms))
    value = job_bytes / MIB / (res_step / 1e3)

    # ---------------- the timed loop: W warm-up + K steps through the reference ABI on pinned host buffers
    for _ in range(args.warmup):
        e2e_step(job)
    for s in job.states:
        s.stats_reset()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    kept = [] if args.dump_outputs and rank == 0 else None
    e2e_ms = [e2e_step(job, kept if i == args.steps - 1 else None) for i in range(args.steps)]
    clocks = sampler.stop() if rank == 0 else None
    if kept is not None:
        dump_outputs(args.dump_outputs, job.comp, np.concatenate(kept),
                     np.concatenate([p[:len(b)].numpy() for p, b in zip(job.pinned, job.blocks)]))
    e2e_step_ms = reduce_max(sum(e2e_ms)) / args.steps
    e2e_val = job_bytes / MIB / (e2e_step_ms / 1e3)
    launches = sum(s.launches() for s in job.states)
    stage_enc = [s.stage_ms(False) for s in job.states]
    stage_dec = [s.stage_ms(True) for s in job.states]
    h2d = total + sum(job.comp)
    d2h = sum(job.comp) + total

    # ---------------- isolated suffix-sort leg: one block alone on the device, radix passes bracketed by CUDA events
    sa_leg = None
    if rank == 0:
        st0 = job.states[0]
        tmp_out = np.zeros(len(job.blocks[0]) + 64, np.uint8)
        for rep in range(4):
            if rep == 1:
                st0.stats_reset()
            flush.fill_(1)
            torch.cuda.synchronize()
            L.bz3_b200_stage_bwt(st0.handle, refs.ptr(job.blocks[0]), len(job.blocks[0]), refs.ptr(tmp_out))
        rec, rounds, sms = C.c_uint64(0), C.c_int32(0), C.c_double(0)
        L.bz3_b200_last_sort_stats(st0.handle, C.byref(rec), C.byref(rounds), C.byref(sms))
        sa_leg = {"records_x_passes": rec.value / 3, "sort_ms": sms.value / 3, "rounds": rounds.value,
                  "block_bytes": len(job.blocks[0])}

    # ---------------- CPU baseline (rank 0, N = 1 only): the reference's pthread path on the same bytes, one round trip
    cpu = None
    if rank == 0 and world == 1:
        try:
            te, td, kind, used = reference_roundtrip(job.blocks, job.bs, reference_jobs())
            cpu = {"value": round(total / MIB / (te + td), 3), "unit": "MiB/s", "cores": used, "kind": kind,
                   "sample": f"one round trip of the whole workload ({nb} blocks, {total} B) with the reference's "
                             f"bz3_encode_blocks/bz3_decode_blocks: {used} pthreads (one per block; -j min(cores, 64) = "
                             f"{reference_jobs()} of {host_threads()} usable host cores)",
                   "encode_MiB_per_s": round(total / MIB / te, 3), "decode_MiB_per_s": round(total / MIB / td, 3)}
        except Exception as ex:  # the CPU leg must never take the GPU numbers down with it
            cpu = {"value": None, "unit": "MiB/s", "cores": 0, "kind": "unavailable", "sample": repr(ex)}

    dev_state_bytes = int(L.bz3_b200_device_bytes(job.states[0].handle))
    dev_ws_bytes = int(L.bz3_b200_workspace_bytes(job.states[0].handle))
    job.close()

    # ---------------- the metric's own configuration: 256 MiB blocks (1 warm-up + 1 timed step)
    headline = None
    late = time.time() - T_START > float(os.environ.get("BZ3_BENCH_HEADLINE_DEADLINE_S", "480"))
    go = (not args.no_headline) and args.workload != HEADLINE and not late
    if dist:  # uniform decision
        t = torch.tensor([1.0 if go else 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        go = t.item() > 0.5
    if go:
        hj = Job(HEADLINE, rank, torch, L, bzip3_b200, refs)
        hb = reduce_sum(hj.total)
        hgate = gated_roundtrip(hj)   # the warm-up step (also sizes the stage workspaces for 256 MiB blocks)
        for s in hj.states:
            s.stats_reset()
        hms = reduce_max(e2e_step(hj))
        hstage_e = [s.stage_ms(False) for s in hj.states]
        hstage_d = [s.stage_ms(True) for s in hj.states]
        headline = {"workload": HEADLINE, "description": WORKLOADS[HEADLINE]["desc"], "blocks_per_gpu": hj.nb,
                    "bytes_per_gpu": hj.total, "steps": 1, "warmup": 1, "ms_per_step": round(hms, 1),
                    "e2e_roundtrip_MiB_per_s": round(hb / MIB / (hms / 1e3), 3), "bit_exact": hgate,
                    "stage_ms": {"encode": {k: round(sum(d[k] for d in hstage_e), 1) for k in bzip3_b200.STAGES},
                                 "decode": {k: round(sum(d[k] for d in hstage_d), 1) for k in bzip3_b200.STAGES},
                                 "note": "summed over the rank's concurrently running blocks"}}
        if rank == 0 and world == 1:
            try:
                te, td, kind, used = reference_roundtrip(hj.blocks, hj.bs, reference_jobs(), check=False)
                headline["cpu_reference"] = {"roundtrip_MiB_per_s": round(hj.total / MIB / (te + td), 3), "threads": used,
                                             "encode_MiB_per_s": round(hj.total / MIB / te, 3),
                                             "decode_MiB_per_s": round(hj.total / MIB / td, 3), "kind": kind}
            except Exception as ex:
                headline["cpu_reference"] = {"error": repr(ex)}
        hj.close()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        traffic = {}
        try:  # DRAM bytes per launch of the dominant kernels, from the committed ncu capture (profiles/README.md)
            traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        except (OSError, ValueError):
            pass

        def stage_total(st, name):
            return sum(d[name] for d in st)

        # dominant kernel = the CM coder of the slower direction; one launch per block per step
        cm_dec_ms = stage_total(stage_dec, "cm") / (nb * args.steps)
        cm_enc_ms = stage_total(stage_enc, "cm") / (nb * args.steps)
        avg_n = total / nb
        avg_c = sum(gate_comp) / nb
        dom = "cm_decode_kernel" if cm_dec_ms >= cm_enc_ms else "cm_encode_kernel"
        dom_ms = max(cm_dec_ms, cm_enc_ms)
        dom_bytes = avg_n + avg_c  # SURVEY 8(d): the coder reads/writes the BWT bytes once and the payload once
        achieved = dom_bytes / (dom_ms / 1e3) / 1e9 if dom_ms > 0 else 0.0
        tr = traffic.get(dom, {}).get(args.workload)
        sa_rec_bytes = float(traffic.get("sa_radix_bytes_per_record", 24.0))
        sa_bytes = sa_rec_bytes * sa_leg["records_x_passes"]
        sa_ach = sa_bytes / (sa_leg["sort_ms"] / 1e3) / 1e9 if sa_leg["sort_ms"] > 0 else 0.0
        whole = (16.0 * total + sum(gate_comp)) * 2 / (e2e_step_ms / 1e3) / 1e9
        out = {
            "metric": "roundtrip_MiB_per_s", "value": round(value, 3), "unit": "MiB/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(e2e_step_ms, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": args.workload, "description": job.w["desc"], "block_size": job.bs, "blocks_per_gpu": nb,
                       "bytes_per_gpu": total, "parallelism": f"blocks sharded {world} way(s), one stream per block",
                       "l2": "256 MiB flush buffer written before every timed step; block buffers + shared stage workspaces >> 126 MB L2",
                       "timed_loop": "the K steps are the e2e path (reference ABI, pinned host buffers); `value` is the device-resident "
                                     "round trip from a side loop of W + K steps (the two differ by the PCIe copies only)",
                       "value_steps": args.steps, "value_ms_per_step": round(res_step, 3),
                       "bit_exact": gate,
                       "hbm_bytes": {"per_block_state": dev_state_bytes, "shared_stage_workspaces": dev_ws_bytes,
                                     "stage_workspaces": int(os.environ.get("BZ3_B200_ARENAS", "2"))},
                       "definition": "one step = encode + decode of every block; throughput = uncompressed bytes / step time"},
            "encode_MiB_per_s": round(job_bytes / MIB / (res_enc / 1e3), 3),
            "decode_MiB_per_s": round(job_bytes / MIB / (res_dec / 1e3), 3),
            "compressed_bytes_rank0": int(sum(gate_comp)),
            "e2e": {"value": round(e2e_val, 3), "unit": "MiB/s", "ms_per_step": round(e2e_step_ms, 3), "steps": args.steps,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "api": "bz3_encode_blocks + bz3_decode_blocks on pinned host buffers"
                           + (" + NCCL gather of compressed blocks to rank 0 (bzip3_b200/sharding.py)" if world > 1 else "")},
            "gpu_launches": int(launches),
            "roofline": {"kernel": dom, "bound": "hbm", "achieved": round(achieved, 6), "peak": hbm_peak, "unit": "GB/s",
                         "frac": round(achieved / hbm_peak, 9), "traffic": tr, "peak_source": peak_src,
                         "note": "serial range-coder recurrence: latency-bound, not bandwidth-bound (DESIGN.md); traffic = "
                                 "dram__bytes_read.sum + dram__bytes_write.sum per launch from profiles/ncu_traffic.json",
                         "avg_launch_ms": round(dom_ms, 3), "algorithmic_bytes_per_launch": int(dom_bytes)},
            "roofline_sa_radix": {"kernel": traffic.get("sa_radix_kernel", "radix passes of the suffix sort"),
                                  "bound": "hbm", "achieved": round(sa_ach, 3), "peak": hbm_peak, "unit": "GB/s",
                                  "frac": round(sa_ach / hbm_peak, 6), "bytes_per_record_per_pass": sa_rec_bytes,
                                  "algorithmic_bytes": int(sa_bytes), "ms": round(sa_leg["sort_ms"], 3),
                                  "rounds": sa_leg["rounds"], "block_bytes": sa_leg["block_bytes"],
                                  "traffic": traffic.get("sa_radix_traffic"),
                                  "note": "one block alone on the device; CUDA events around every radix sort of the suffix "
                                          "sorter (no host sync inside)"},
            "roofline_whole_job": {"achieved": round(whole, 3), "peak": hbm_peak, "unit": "GB/s",
                                   "frac": round(whole / hbm_peak, 9), "note": "SURVEY 8(d): (16 n + c) bytes per direction"},
            "stage_ms_per_step": {"encode": {k: round(stage_total(stage_enc, k) / args.steps, 3) for k in bzip3_b200.STAGES},
                                  "decode": {k: round(stage_total(stage_dec, k) / args.steps, 3) for k in bzip3_b200.STAGES},
                                  "note": "summed over the rank's concurrently running blocks"},
            "headline_b256": headline,
            "cpu_baseline": cpu,
            "clocks": clocks,
        }
        _emit(out)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def _quiet_stdout():
    """Libraries (NCCL's version banner, torchrun notices) write to fd 1; the contract is ONE JSON line on stdout.
    Point fd 1 at stderr for the duration of the run and keep the real stdout for the result line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def _emit(obj):
    line = json.dumps(obj)
    if _REAL_STDOUT is not None:
        _REAL_STDOUT.write(line + "\n")
        _REAL_STDOUT.flush()
    else:
        print(line, flush=True)


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("BZ3_BENCH_WORKLOAD", "zipf100m_b16"), choices=sorted(WORKLOADS))
    ap.add_argument("--no-headline", action="store_true", help="skip the 256 MiB-block sub-record")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0's compressed block sizes, compressed bytes and "
                         "decoded bytes) to DIR/<name>.npy; the compressed blocks are copied aside inside that step")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
    else:
        run_b200_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
