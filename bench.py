#!/usr/bin/env python
"""bench.py -- input MiB/s of ZopfliCompress(gzip, numiterations=15, blocksplittingmax=15).

A "step" is one whole compression of the workload: config C2 of BASELINE.json (100,000,000 B of
enwik8-like text, numiterations=15) per GPU.  With N>1 (torchrun, one rank per GPU) the job is ONE gzip
stream over ONE input of N x 100 MB held by rank 0: the library itself (zopfli_b200/csrc/dist.cpp) scatters
the master-block shards over NCCL, every rank compresses its shard, and the compressed bits are gathered
straight into their final bit positions on rank 0 (SURVEY 8(e)).  Weak scaling: per-GPU work is fixed.

  value   whole-job MiB/s with the input already resident in HBM when the timed region starts
  e2e     the same through the reference-facing C ABI with a PAGEABLE host buffer (H2D + D2H inside)
  --impl reference   the reference's own CPU implementation (oracle/_ref) on a bounded sample
  --dump-outputs DIR after the timed steps, the last step's gzip stream as .npy files (see dump_outputs)
"""
import argparse
import gzip
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import zref  # noqa: E402

MIB = float(1 << 20)
MB = 1_000_000               # master block (util.h:60)
SHARD = 100_000_000          # config C2 per GPU
NUMITER = 15
ALG_BYTES_PER_STEP = 34.0    # SURVEY 8(d): 28 table + 1 input + 2+2 length_array + ~0.6 store, per position-iteration
REF_MASTERS = 8              # master blocks the CPU reference is timed on (K >= 8, BASELINE.md 3.3)
GIANT_MASTERS = [85, 84, 78, 42, 40]            # master blocks of the C2 text with the largest deflate blocks
UNIFORM_MASTERS = [3, 15, 27, 39, 51, 63, 75, 99]  # (tools/find_giant_masters.py)


WORKLOAD = "c2"   # c2 (default, the metric's config) | c3 (1 GiB, strong scaling) | c4 (binary, 50 iterations)
SCALING = "weak"


def select_workload(name, world):
    """BASELINE.json configs: C2 = 100 MB text per GPU at 15 iterations (the bench line the driver reads);
    C3 = one 1 GiB text stream over 1/2/4/8 GPUs (strong scaling: the same bytes at every N);
    C4 = 51,220,480 B of redundant binary at 50 iterations on one GPU."""
    global WORKLOAD, SHARD, NUMITER, SCALING, REF_MASTERS
    WORKLOAD = name
    if name == "c3":
        assert (1 << 30) % world == 0 and 8 % world == 0
        SHARD, NUMITER, SCALING = (1 << 30) // world, 15, "strong"
    elif name == "c4":
        assert world == 1
        SHARD, NUMITER, REF_MASTERS = 51220480, 50, 2
    elif name != "c2":
        raise SystemExit("unknown workload " + name)


def segment(rank, world):
    """this rank's part of the one input (rank 0 assembles the parts in rank order)"""
    from zopfli_b200 import corpus
    if WORKLOAD == "c3":   # eight fixed 128 MiB segments (seeds 3..10), 8 / world of them per rank
        per = 8 // world
        return b"".join(corpus.synth_text(1 << 27, 3 + rank * per + k) for k in range(per)), "synthetic"
    if WORKLOAD == "c4":
        return corpus.synth_binary(SHARD, 4), "synthetic"
    return workload(SHARD, 2 + rank)


def bench_config(world):
    if WORKLOAD == "c3":
        what = "C3 web-text-like, 1073741824 B in one stream (%d B per GPU), gzip, numiterations=15, blocksplittingmax=15" % SHARD
    elif WORKLOAD == "c4":
        what = "C4 redundant binary, %d B, gzip, numiterations=50, blocksplittingmax=15" % SHARD
    else:
        what = ("C2 enwik8-like text, %d B per GPU (%d B total, one stream), gzip, numiterations=15, "
                "blocksplittingmax=15" % (SHARD, SHARD * world))
    return {"workload": what,
            "l2": "inputs and working set (GBs) far larger than the 126 MB L2; no flush needed",
            "parallelism": "master-block shards x%d inside the library: NCCL scatter of byte ranges, NCCL gather of "
                           "compressed bits at their final bit offsets" % world if world > 1
            else "single GPU, all blocks of all master blocks in flight"}


def workload(nbytes, seed):
    path = os.environ.get("ZOPFLI_BENCH_ENWIK8")
    if path and os.path.exists(path) and seed == 2:
        return open(path, "rb").read()[:nbytes], "file:" + os.path.basename(path)
    from zopfli_b200 import corpus
    return corpus.synth_text(nbytes, seed), "synthetic"


class ClockSampler(threading.Thread):
    def __init__(self, dev):
        super().__init__(daemon=True)
        self.dev, self.stop_flag, self.sm, self.maxsm, self.reasons = dev, False, [], 0, set()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.sm.append(float(o[0]))
                self.maxsm = float(o[1])
                for n, v in zip(names, o[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.maxsm or None,
                "reasons": sorted(self.reasons)}


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("k_iterate_bytes_per_launch")
        except Exception:
            pass
    return None


# ---- the reference on the host cores (oracle/_ref: the unmodified reference, -O3 -DNDEBUG, 1 thread) ----

def cpu_reference(data, masters, steps, warmup):
    """times ZopfliCompress(gzip) of the first `masters` master blocks; the reference has no threading"""
    import zref
    ref = zref.Ref(ndebug=True)
    sample = data[:masters * MB]
    for _ in range(warmup):
        ref.compress(data[:MB], 0, numiterations=NUMITER)  # warm-up: code and tables paged in
    times, out = [], None
    for _ in range(steps):
        t = time.perf_counter()
        out = ref.compress(sample, 0, numiterations=NUMITER)
        times.append(time.perf_counter() - t)
    sec = sum(times) / len(times)
    return len(sample) / MIB / sec, sec, out


def _ref_part(args):
    import zref
    piece, s, e, final = args
    return zref.Ref(ndebug=True).deflate_part(piece, s, e, final=final, numiterations=NUMITER)


def reference_parts(data, masters, nmasters_total):
    """ZopfliDeflatePart of sampled master blocks: the reference itself in a process pool (the children never
    touch CUDA) where oracle/_ref is built, its recorded answers (tests/golden/reference_answers.json) elsewhere"""
    jobs = []
    for m in masters:
        a, b = m * MB, min(len(data), (m + 1) * MB)
        lo = max(0, a - 32768)
        jobs.append((data[lo:b], a - lo, b - lo, int(m == nmasters_total - 1)))
    if not zref.reference_built(ndebug=True):
        return zref.reference().map("deflate_part", jobs, numiterations=NUMITER)
    with mp.get_context("fork").Pool(min(8, max(1, len(jobs)))) as pool:
        return pool.map(_ref_part, jobs)


def bits_of(b):
    return np.unpackbits(np.frombuffer(b, dtype=np.uint8), bitorder="little")


def dump_outputs(path, stream):
    """The last timed step's result, the gzip stream a caller receives, as float32/float64 .npy files under 64 MB:
    its length, and its byte values at a fixed seeded sample of at most 4 Mi positions (all of them if shorter)."""
    os.makedirs(path, exist_ok=True)
    a = np.frombuffer(stream, dtype=np.uint8)
    idx = np.arange(len(a)) if len(a) <= (4 << 20) else \
        np.sort(np.random.default_rng(0).choice(len(a), 4 << 20, replace=False))
    np.save(os.path.join(path, "gzip_length.npy"), np.array([len(a)], dtype=np.float64))
    np.save(os.path.join(path, "gzip_sample_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, "gzip_sample_bytes.npy"), a[idx].astype(np.float32))


def check_against_reference(stream, offs, data, masters, prefix_out=None, prefix_masters=0):
    """Sampled master blocks of `stream` (a gzip file) == the reference's ZopfliDeflatePart of the same
    ranges, located through the per-master-block bit offsets; plus, if given, the reference's gzip of the
    first `prefix_masters` master blocks as a bit prefix.  Returns (bytes covered, identical)."""
    body = bits_of(stream[10:-8])
    nm = len(offs) - 1
    ok, covered = True, 0
    if prefix_out is not None and prefix_masters > 1:
        pb = bits_of(prefix_out[10:-8])
        n = int(offs[prefix_masters - 1])  # the last block of the sample carries BFINAL there, not here
        ok &= bool(np.array_equal(body[:n], pb[:n]))
        covered += (prefix_masters - 1) * MB
    want = reference_parts(data, masters, nm)
    for m, w in zip(masters, want):
        # the master block's bits zero-padded to whole bytes, and its bit count mod 8: ZopfliDeflatePart's (bytes, bp)
        got = np.packbits(body[offs[m]:offs[m + 1]], bitorder="little").tobytes(), int(offs[m + 1] - offs[m]) & 7
        ok &= bool(got == w)
        covered += min(len(data), (m + 1) * MB) - m * MB
    return covered, ok


def run_reference(args, rank):
    if rank != 0:
        return
    data, kind = segment(0, 1) if WORKLOAD != "c2" else workload(SHARD, 2)
    steps, warmup = args.steps, args.warmup
    # the whole run is bounded to a few minutes: ~1.6 s of CPU per master block
    masters = min(REF_MASTERS, max(2, int(150 / max(1, steps))))
    v, sec, _ = cpu_reference(data, masters, steps, warmup)
    sample = ("first %d bytes (%d master blocks) of the workload per step, oracle/_ref -O3 -DNDEBUG, 1 thread "
              "(the reference has no threading); warm-up steps use 1 master block" % (masters * MB, masters))
    line = {"impl": "reference", "metric": "input MiB/s at numiterations=%d" % NUMITER, "value": v, "unit": "MiB/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": SCALING, "vs_baseline": None, "dtype": "u8", "data": kind,
            "config": bench_config(args.gpus),
            "cpu_baseline": {"value": v, "unit": "MiB/s", "cores": 1, "kind": "reference", "sample": sample},
            "e2e": {"value": v, "unit": "MiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_product(args, rank, world):
    os.environ.setdefault("NCCL_DEBUG", "WARN")
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's version banner must not land on stdout: one JSON line only
    import torch
    import torch.distributed as dist
    import zopfli_b200 as zb

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    os.environ["ZOPFLI_B200_DEVICE"] = str(local)
    lib = zb.library()
    steps, warmup = args.steps, args.warmup

    # ---- the workload: rank r generates segment r (seed 2 + r); rank 0 assembles the one input ----
    seg, kind = segment(rank, world)
    n_total = SHARD * world
    if world > 1:
        mine = torch.frombuffer(bytearray(seg), dtype=torch.uint8).to(dev)
        parts = [torch.empty(SHARD, dtype=torch.uint8, device=dev) for _ in range(world)] if rank == 0 else None
        dist.gather(mine, parts, dst=0)
        data = b"".join(p.cpu().numpy().tobytes() for p in parts) if rank == 0 else None
        del mine, parts
        # the library's own communicator (csrc/dist.cpp); the id travels through torch.distributed
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(lib.dist_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        # NCCL prints its version banner with printf when a communicator is created (NCCL_DEBUG=WARN):
        # stdout carries exactly one JSON line, so fd 1 points at stderr while the library initialises
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            lib.dist_init(rank, world, idt.cpu().numpy().tobytes())
        finally:
            os.dup2(saved, 1)
            os.close(saved)
    else:
        data = seg
    # pageable host copy (what a drop-in C caller passes); +64 so the device-resident leg can share it
    host = np.zeros(n_total + 64, dtype=np.uint8) if rank == 0 else np.zeros(64, dtype=np.uint8)
    if rank == 0:
        host[:n_total] = np.frombuffer(data, dtype=np.uint8)
    hptr = host.ctypes.data
    devbuf = None
    if world == 1:
        devbuf = torch.zeros(n_total + 64, dtype=torch.uint8, device=dev)
        devbuf[:n_total].copy_(torch.from_numpy(host[:n_total]))
        torch.cuda.synchronize()

    def job(resident):
        """one whole compression; rank 0 gets the library's malloc()ed gzip stream (no copy into Python)"""
        if world == 1:
            return lib.compress_ptr_nocopy(hptr, n_total, zb.ZOPFLI_FORMAT_GZIP,
                                           dev_ptr=devbuf.data_ptr() if resident else None, numiterations=NUMITER)
        return lib.dist_compress_ptr_nocopy(hptr, n_total, zb.ZOPFLI_FORMAT_GZIP, staged=resident, numiterations=NUMITER)

    def timed(resident):
        if world > 1 and resident:  # stage the shards once, outside the timed region
            w = job(False)
            if w is not None:
                w.close()
        for _ in range(warmup):
            w = job(resident)
            if w is not None:
                w.close()
        lib.reset_stats()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler = ClockSampler(local)
        sampler.start()
        t0 = time.perf_counter()
        e0.record()
        out = None
        for _ in range(steps):
            if out is not None:
                out.close()
            out = job(resident)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        wall = time.perf_counter() - t0
        sampler.stop_flag = True
        # every call ends with the synchronous device->host copy of the stream, so the host clock brackets
        # the device work; the library's kernels run on its own streams (CUDA events there feed `stats`)
        ms = max(e0.elapsed_time(e1), wall * 1e3)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        st = lib.stats()
        offs = lib.last_master_bit_offsets() if world == 1 else None
        if out is not None:
            buf, out = out, out.tobytes()  # outside the timed region: only the checks below need a bytes object
            buf.close()
        return float(t.item()) / steps, out, st, sampler.summary(), offs

    ms_res, out_res, st_res, clocks, offs = timed(True)
    ms_e2e, out_e2e, st_e2e, _, _ = timed(False)
    if rank == 0:
        assert out_res == out_e2e, "resident and host-buffer runs disagree"
        assert gzip.decompress(out_res) == data, "output does not inflate to the input"
        nm = (n_total + MB - 1) // MB
        cpu = None
        if world == 1:
            ref_out = None   # the CPU baseline needs the reference itself (oracle/_ref), not its recorded answers
            if zref.reference_built(ndebug=True):
                cpu_v, cpu_sec, ref_out = cpu_reference(data, REF_MASTERS, 1, 0)
                cpu = {"value": cpu_v, "unit": "MiB/s", "cores": 1, "kind": "reference",
                       "sample": "first %d bytes (%d master blocks) of the workload, oracle/_ref -O3 -DNDEBUG, 1 thread "
                                 "(the reference has no threading)" % (REF_MASTERS * MB, REF_MASTERS)}
            masters = GIANT_MASTERS + UNIFORM_MASTERS if (kind == "synthetic" and WORKLOAD == "c2") else \
                list(range(REF_MASTERS, nm, max(1, nm // 13)))[:13]
            covered, same = check_against_reference(out_res, offs, data, masters, ref_out, REF_MASTERS)
            check = {"sample_bytes": covered, "identical": bool(same), "delta_bytes_vs_reference": 0 if same else None,
                     "how": ("timed output vs reference: bit prefix of the first %d master blocks + " % (REF_MASTERS - 1)
                             if ref_out is not None else "timed output vs the reference's recorded answers: ") +
                            "ZopfliDeflatePart of master blocks %s (incl. the five largest blocks), located by bit "
                            "offsets" % masters}
        else:
            # the N-GPU stream must be the single-GPU stream of the same input (itself reference-checked above
            # and in tests/), and sampled master blocks of every rank's shard are compared with the reference
            single = lib.compress_ptr_nocopy(hptr, n_total, zb.ZOPFLI_FORMAT_GZIP, numiterations=NUMITER)
            offs1 = lib.last_master_bit_offsets()
            single_bytes = single.tobytes()
            single.close()
            per = nm // world
            masters = sorted(set([r * per for r in range(world)] + [r * per + per // 2 for r in range(world)] + [nm - 1]))
            covered, same = check_against_reference(out_res, offs1, data, masters)
            check = {"sample_bytes": covered, "identical": bool(same and single_bytes == out_res),
                     "equals_single_gpu_stream": single_bytes == out_res, "inflates_to_input": True,
                     "how": "N-GPU stream == 1-GPU stream of the same input; master blocks %s vs reference ZopfliDeflatePart" % masters}
        peak, peak_src = peak_hbm()
        # k_iterate runs as several concurrent launches per step (chunk pipelines x {giant blocks, the rest},
        # fixed-tree re-parses); ms_iterate is the sum of their CUDA-event durations on their own streams
        nl = max(1, int(st_res["iterate_launches"]))
        it_s = st_res["ms_iterate"] / 1e3 / nl                            # average launch duration
        alg = ALG_BYTES_PER_STEP * st_res["iterate_steps"] / nl          # algorithmic bytes of an average launch
        achieved = alg / it_s / 1e9 if it_s > 0 else 0.0
        traffic = ncu_traffic()
        sm_mhz = clocks.get("sm_mhz") or 1965.0
        cyc = st_res["cyc_max"]
        maxpos = int(st_res["max_block_positions"])
        line = {"metric": "input MiB/s at numiterations=%d" % NUMITER, "value": n_total / MIB / (ms_res / 1e3), "unit": "MiB/s",
                "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_res, "higher_is_better": True,
                "scaling": SCALING, "vs_baseline": None, "dtype": "u8", "data": kind,
                "config": bench_config(world),
                "e2e": {"value": n_total / MIB / (ms_e2e / 1e3), "unit": "MiB/s", "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": st_e2e["h2d_bytes"] / steps,
                        "d2h_bytes_per_step": st_e2e["d2h_bytes"] / steps, "host_buffer": "pageable"},
                "gpu_launches": int(st_res["launches"]),
                "clocks": clocks,
                "roofline": {"bound": "hbm", "kernel": "k_iterate", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": traffic,
                             "traffic_over_algorithmic": (traffic / alg) if traffic and alg else None,
                             "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg, "launch_ms": it_s * 1e3,
                             "launches_per_step": nl / steps,
                             # BASELINE.md 3.5: the bound that matters is the DP dependency chain of the largest block
                             "chain_bound_ms": sum(cyc) / sm_mhz / 1e3,
                             "chain": {"max_block_positions": maxpos, "iterations": NUMITER,
                                       "dp_cycles_per_step": cyc[1] / max(1, maxpos * NUMITER),
                                       "all_cycles_per_step": sum(cyc) / max(1, maxpos * NUMITER),
                                       # share of all DP steps of the step that ran in the integer window (iterate.cuh)
                                       "integer_window_share": st_res.get("int_steps", 0) / max(1, st_res["iterate_steps"])},
                             "note": "DP dependency chain, not bandwidth, bounds this kernel (SURVEY 7.2 #5): "
                                     "chain_bound_ms = cycles of the critical block / SM clock"},
                "cpu_baseline": cpu,
                "parity": check,
                "output_bytes": len(out_res),
                "kernel_ms_per_step": {k: v / steps for k, v in st_res.items() if k.startswith("ms_")}}
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, out_res)
    if world > 1:
        dist.barrier()
        lib.dist_finalize()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="c2", help="c2 (default) | c3 (1 GiB, strong scaling) | c4 (binary, 50 iterations)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output there as .npy files")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    select_workload(args.workload, world)
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_product(args, rank, world)


if __name__ == "__main__":
    main()
