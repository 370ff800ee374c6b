#!/usr/bin/env python
"""bench.py -- headline benchmark for the block-level aggregation hot path.

A "step" is ONE pass of the aggregator over one synthetic vector set:
  workload c3 (default; the config BASELINE.json's target is quoted on, configs[2]):
      bm::aggregator::combine_and_sub over 1024 vectors x 2^30 bits, Zipf density mix d_k = 0.5/k,
      every vector optimize()d (k <~ 51 bit-blocks, the rest GAP), AND = {1,2}, SUB = {3..1024}, opt_compress
  workload c2 (configs[1]): combine_or over 256 vectors x 2^28 bits, 5 % density, bit-blocks only
  workload c5 (configs[4]): one GPU's shard of combine_or over 4096 vectors x 2^32 bits sharded over 8 GPUs
Multi-GPU (torchrun, one rank per GPU): the block range is sharded -- every rank owns a contiguous range of block columns of
every vector (weak scaling: a full-size shard per rank), aggregates it locally, and the ranks exchange per-block popcounts +
cardinalities with ONE ncclAllGather issued by the library itself (bmb200_exchange_popcounts) on a side stream, so the
exchange of step i overlaps the kernel of step i+1.  torch.distributed only carries the barrier / max-over-ranks plumbing.

What one run reports (one JSON line):
  value / roofline  device-resident aggregation, CUDA events on the launching stream
  parity            ALL result columns (kind, popcount, digest, GAP length) against the unmodified reference running on the
                    host cores over inputs regenerated on the HOST by an independent implementation of the generator
  e2e               through bm::b200::aggregator on REAL bm::bvector<> objects (oracle/_ref/libbmb200_e2e.so): cold =
                    tree walk + pack + H2D + kernel + D2H + result bvector every step (the contract's e2e), warm = sources
                    resident in a bm::b200::device_set (upload once), split of the cold step, result compared with bm::aggregator
  cpu_baseline      the reference on 1 thread (bounded sample) and on all cores (whole workload)

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c3|c2|c5] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned to its caller (rank 0's shard) as float64 .npy files, so that two
builds can be compared output for output on identical (seeded) inputs: per result column kind, popcount, digest (two 32-bit
halves), GAP run count, the total, and the 2048 result words of a fixed, seeded sample of columns (GAP columns expanded).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

WORKLOADS = {
    "c3": dict(n_vec=1024, n_blocks=16384, op="and_sub", desc="combine_and_sub 1024 x 2^30 bits, Zipf d_k=0.5/k, optimize()d (bit + GAP), AND={1,2} SUB={3..1024}, opt_compress"),
    "c2": dict(n_vec=256, n_blocks=4096, op="or", desc="combine_or 256 x 2^28 bits, iid 5% density, bit-blocks"),
    # configs[4]: 4096 x 2^32 bits block-range sharded over 8 GPUs = 8192 block columns per GPU; density is not fixed by
    # BASELINE (as bit-blocks it would be 2 TiB), SURVEY 8d proposes iid p=0.0025 + optimize() => GAP blocks, ~22 GB per GPU
    "c5": dict(n_vec=4096, n_blocks=8192, op="or", desc="combine_or 4096 vectors, 8192 block columns per GPU (2^32 bits over 8 GPUs), iid 0.25% density, optimize()d (GAP blocks)"),
}
OPS = {"or": 0, "and": 1, "and_sub": 2}
F_OPT_NONE, F_OPT_COMPRESS = 0, 2


def workload_inputs(name: str, rank: int):
    w = WORKLOADS[name]
    nv = w["n_vec"]
    if name == "c3":
        dens = np.array([0.5 / (k + 1) for k in range(nv)])
        seed = np.arange(1000, 1000 + nv, dtype=np.uint64) + np.uint64(1_000_003 * rank)
        optimize = True
    elif name == "c5":
        dens = np.full(nv, 0.0025)
        seed = np.arange(5000, 5000 + nv, dtype=np.uint64) + np.uint64(1_000_003 * rank)
        optimize = True
    else:
        dens = np.full(nv, 0.05)
        seed = np.arange(100, 100 + nv, dtype=np.uint64) + np.uint64(1_000_003 * rank)
        optimize = False
    return dens, seed, optimize


def workload_groups(name: str):
    nv = WORKLOADS[name]["n_vec"]
    if name == "c3":
        return OPS["and_sub"], np.array([0, 1], np.uint32), np.arange(2, nv, dtype=np.uint32), F_OPT_COMPRESS
    if name == "c5":
        return OPS["or"], np.arange(nv, dtype=np.uint32), None, F_OPT_COMPRESS
    return OPS["or"], np.arange(nv, dtype=np.uint32), None, F_OPT_NONE


def cpu_model() -> str:
    try:
        return next(ln.split(":", 1)[1].strip() for ln in open("/proc/cpuinfo") if ln.startswith("model name"))
    except Exception:
        return "unknown"


def mem_available_gb() -> float:
    try:
        return int(next(ln for ln in open("/proc/meminfo") if ln.startswith("MemAvailable")).split()[1]) / 2**20
    except Exception:
        return 1e9


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines: list[str] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled_traffic(workload: str):
    """dram__bytes_read+write per launch of the dominant kernel from the newest committed ncu capture (profiles/), or None."""
    key = {"c3": "c3_agg_kernel_and_sub", "c2": "c2_agg_kernel_or", "c5": "c5_agg_kernel_or"}.get(workload)
    for rnd in ("r02", "r01"):
        f = ROOT / "profiles" / rnd / "ncu_agg_kernel.json"
        try:
            d = json.loads(f.read_text())[key]

            def gb(x):
                return float(x["value"]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[x["unit"]]
            return int(gb(d["dram__bytes_read.sum"]) + gb(d["dram__bytes_write.sum"])), f"profiles/{rnd}/ncu_agg_kernel.json (ncu --set full, same command, full-size shard)"
        except Exception:
            continue
    return None, None


def device_set_stats(ctx, dset, torch):
    """Count source blocks by kind and the exact GAP payload with a few torch ops over the device arrays."""
    ptrs = dset.device_ptrs()
    n = dset.n_vec * dset.n_blocks

    class Wrap:
        def __init__(self, addr, nbytes, typestr, shape):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (addr, False), "version": 2}
    desc = torch.as_tensor(Wrap(ptrs.desc, n * 4, "<i4", (n,)), device=f"cuda:{ctx.device}").long() & 0xFFFFFFFF
    kind = desc & 3
    counts = {"null": int((kind == 0).sum()), "full": int((kind == 1).sum()), "bit": int((kind == 2).sum()), "gap": int((kind == 3).sum())}
    gap_words = 0
    if counts["gap"]:
        gp = torch.as_tensor(Wrap(ptrs.gap_pool, dset.n_gap_units * 16, "<i2", (dset.n_gap_units * 8,)), device=f"cuda:{ctx.device}")
        gb = torch.as_tensor(Wrap(ptrs.gap_base, (dset.n_blocks + 1) * 8, "<i8", (dset.n_blocks + 1,)), device=f"cuda:{ctx.device}")
        col = torch.arange(dset.n_blocks, device=desc.device).repeat_interleave(dset.n_vec)
        isgap = kind == 3
        dg = desc[isgap]
        off = (gb[col[isgap]] + ((dg >> 2) & 0x0FFFFFFF)) * 8 + (dg >> 31)      # + lead pad (BMB200_DESC_GAP_PAD)
        hdr = gp[off].long() & 0xFFFF
        gap_words = int(((hdr >> 3) + 1).sum())
    return counts, gap_words


# ----------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    """--impl reference: the UNMODIFIED reference (oracle/_ref/libbmref*.so, compiled from /root/reference/src) on the host cores.
    Inputs come from the host restatement of the generator (oracle/bm_synth.c): no GPU, no product library in this process.
    The bvectors are built once; every step is one pass of bm::aggregator over the WHOLE workload on T = nproc worker threads,
    each with its own aggregator over a contiguous range of block columns (BASELINE.md section 3)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    import orclib
    w = WORKLOADS[args.workload]
    n_cols = args.cols or w["n_blocks"]
    cores = os.cpu_count() or 1
    threads = max(1, min(args.ref_threads or cores, n_cols))
    dens, seed, optimize = workload_inputs(args.workload, 0)
    op, g0, g1, flags = workload_groups(args.workload)
    need_gb = 2.3 * (13.5 if args.workload == "c3" else 22.5 if args.workload == "c5" else 8.1) * n_cols / w["n_blocks"]
    if mem_available_gb() < need_gb:
        return {"impl": "reference", "unavailable": f"host has {mem_available_gb():.0f} GB available, the workload needs {need_gb:.0f} GB"}
    t0 = time.time()
    hs = orclib.HostSynth(w["n_vec"], n_cols, dens, seed, optimize, threads=min(cores, 64))
    t_synth = time.time() - t0
    ps = hs.ps
    n_src_blocks = int((ps.kinds() != 0).sum())
    stored = ps.stored_bytes()
    have = orclib.have_ref()
    rows = {}
    # rows: (a) one worker per whole 256-block superblock range, T = min(nproc, superblocks) -- the split the reference's own
    # top-level walk favours; (b) T = nproc workers over finer ranges (BASELINE.md section 3 "all cores"); (c) the AVX-512 build on (a).
    t_sb = max(1, min(threads, n_cols // 256)) if n_cols >= 256 else threads
    configs = [("avx2_sb", False, t_sb)]
    if threads != t_sb:
        configs.append(("avx2_nproc", False, threads))
    if have and orclib.have_ref("avx512") and orclib.cpu_has_avx512():
        configs.append(("avx512_sb", "avx512", t_sb))
    if not have:
        # the C port (oracle/bm_oracle.c), 1 thread -- only when oracle/_ref was not built (no /root/reference at build time)
        t0 = time.perf_counter(); orclib.oracle_aggregate(ps, op, g0, g1, flags, 0, min(n_cols, 256)); sec = time.perf_counter() - t0
        frac = min(n_cols, 256) / n_cols
        rows["port"] = {"ms": 1e3 * sec / frac, "threads": 1, "simd": "scalar", "result_bits": None, "extrapolated_from_cols": min(n_cols, 256)}
    for name, var, thr in configs if have else []:
        t0 = time.time()
        job = orclib.RefJob(ps, op, g0, g1, flags, threads=thr, variant=var)
        t_build = time.time() - t0
        job.run(max(1, args.warmup))
        sec, tot = job.run(args.steps)
        rows[name] = {"ms": 1e3 * float(np.mean(sec)), "ms_min": 1e3 * float(np.min(sec)), "threads": job.threads,
                      "simd": orclib.ref(var).ref_simd().decode(), "result_bits": int(tot), "build_s": round(t_build, 2)}
        job.free()
    best = min(rows, key=lambda k: rows[k]["ms"])
    ms = rows[best]["ms"]
    value = n_src_blocks / (ms * 1e-3)
    kind = "reference" if have else "port"
    sample = f"all {n_cols} block columns x {w['n_vec']} vectors per step ({stored / 2**20:.0f} MiB), bvectors built once"
    hs.free()
    return {"impl": "reference", "metric": "aggregator input 64Kbit-blocks/s", "value": value, "unit": "blocks/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": args.workload + ": " + w["desc"], "sample": sample, "reduced": bool(args.cols and args.cols != w["n_blocks"]),
                       "inputs": f"host generator oracle/bm_synth.c, {t_synth:.1f} s on {min(cores, 64)} threads"},
            "cpu_baseline": {"value": value, "unit": "blocks/s", "cores": rows[best]["threads"], "kind": kind, "sample": sample,
                             "simd": rows[best]["simd"], "nproc": cores, "cpu": cpu_model(), "rows": rows,
                             "gbs": stored / (ms * 1e-3) / 1e9},
            "e2e": {"value": value, "unit": "blocks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "result_bits": rows[best]["result_bits"]}


# ----------------------------------------------------------------------------------------------- parity + e2e helpers
def full_parity(workload, n_cols, rank, res_meta, threads):
    """ALL columns of the GPU result against the unmodified reference over host-generated inputs (rank's own seeds)."""
    import orclib
    w = WORKLOADS[workload]
    dens, seed, optimize = workload_inputs(workload, rank)
    op, g0, g1, flags = workload_groups(workload)
    kind_r, pop_r, dig_r, nr_r = res_meta
    t0 = time.time()
    hs = orclib.HostSynth(w["n_vec"], n_cols, dens, seed, optimize, threads=min(threads, 64))
    t_synth = time.time() - t0
    if n_cols >= 256:
        threads = max(1, min(threads, n_cols // 256))     # whole superblocks per reference worker (see run_reference)
    out = {"cols": int(n_cols), "fields": ["kind", "popcnt", "digest", "gap_len"], "inputs": "regenerated on the host (oracle/bm_synth.c)",
           "host_synth_s": round(t_synth, 2)}
    if orclib.have_ref():
        t0 = time.time()
        job = orclib.RefJob(hs.ps, op, g0, g1, flags, threads=threads)
        t_build = time.time() - t0
        job.run(1)
        sec, tot = job.run(3)
        k, p, d, gl = job.export()
        job.free()
        out.update(against="oracle/_ref/libbmref.so (unmodified reference, bm::aggregator)", ref_threads=int(threads), ref_build_s=round(t_build, 2),
                   ref_ms=1e3 * float(np.mean(sec)), ref_ms_min=1e3 * float(np.min(sec)))
        gap = k == 3
        eq = {"kind": bool(np.array_equal(k, kind_r)), "popcnt": bool(np.array_equal(p, pop_r)), "digest": bool(np.array_equal(d, dig_r)),
              "gap_len": bool(np.array_equal(gl[gap], nr_r[gap]))}
    else:   # GPU box without oracle/_ref (should not happen: the prebuilt files travel): the C port on a bounded range
        nc = min(n_cols, 512)
        k, p, d, nr, _, _ = orclib.oracle_aggregate(hs.ps, op, g0, g1, flags, 0, nc)
        out.update(against="oracle/liboracle.so (C port)", cols=int(nc))
        eq = {"kind": bool(np.array_equal(k, kind_r[:nc])), "popcnt": bool(np.array_equal(p, pop_r[:nc])), "digest": bool(np.array_equal(d, dig_r[:nc])),
              "gap_len": bool(np.array_equal(nr[k == 3], nr_r[:nc][k == 3]))}
    src_blocks = int((hs.ps.kinds() != 0).sum())
    stored = hs.ps.stored_bytes()
    hs.free()
    out["equal"] = all(eq.values())
    out["per_field"] = eq
    return out, src_blocks, stored


class E2E:
    """ctypes face of oracle/_ref/libbmb200_e2e.so (oracle/e2e_harness.cpp): bm::b200::aggregator on real bm::bvector<> objects."""

    def __init__(self, name="libbmb200_e2e.so"):
        so = ROOT / "oracle" / "_ref" / name
        self.lib = C.CDLL(str(so)) if so.exists() else None
        if self.lib:
            self.lib.e2e_create_empty.restype = C.c_void_p
            self.lib.e2e_free.restype = None
        self.h = None

    def ok(self):
        return self.lib is not None


def run_e2e(args, ctx, dset, device, world, dist, torch, op, g0, g1, flags, total_bits, src_blocks_all):
    """cold / warm end-to-end through the C++ binding on real bvectors built from this rank's (downloaded) inputs"""
    from bitmagic_b200.capi import packed_c, ptr
    e = E2E()
    if not e.ok():
        return {"unavailable": "oracle/_ref/libbmb200_e2e.so not built (needs the reference headers at build time)"}
    need_gb = 1.3 * dset.stored_bytes() / 2**30 * world + 8          # every rank of this node keeps its bvectors on the host
    if mem_available_gb() < need_gb:
        return {"unavailable": f"host memory: {mem_available_gb():.0f} GB available, e2e needs {need_gb:.0f} GB for the host bvectors"}
    cores = os.cpu_count() or 1
    thr = max(1, cores // max(1, world))
    if world > 1:       # ranks that share a NUMA node share its cores: size every rank's packer team for its share (half of it, the issuing thread needs a CPU)
        try:
            n_nodes = max(1, len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]))
        except OSError:
            n_nodes = 1
        per_node = -(-world // n_nodes)
        os.environ["BMB200_HOST_THREADS"] = str(max(2, min(32, (cores // n_nodes) // per_node // 2)))
    lib = e.lib
    g1a = g1 if g1 is not None else np.zeros(0, np.uint32)
    node = C.c_int(-1)

    def build_bvectors(lib_):
        # real bm::bvector<> objects, filled chunk by chunk from the device copy of this rank's inputs (the download is setup, not timed)
        h_ = C.c_void_p(lib_.e2e_create_empty(C.c_uint32(dset.n_vec), C.c_uint32(dset.n_blocks), int(device), 1, C.byref(node)))
        assert h_, "e2e_create_empty failed"
        step_cols = 1024
        for lo in range(0, dset.n_blocks, step_cols):
            ps = dset.download(lo, min(dset.n_blocks, lo + step_cols))
            c = packed_c(ps.n_vec, ps.n_blocks, ps.desc, ps.bit_base, ps.gap_base, ps.bit_pool, ps.gap_pool)
            rc_ = lib_.e2e_append(h_, C.byref(c), C.c_uint32(lo), int(min(thr, 64)))
            assert rc_ == 0, "e2e_append failed"
            del ps
        return h_
    h = build_bvectors(lib)
    n0, n1 = int(g0.size), int(g1a.size)
    compress = 1 if flags & F_OPT_COMPRESS else 0

    def sync_all():
        if world > 1:
            dist.barrier()
    # ---- cold: tree walk + pack + H2D + kernel + D2H + bvector, every step ----
    ms = np.zeros(args.e2e_steps + 1); cnt = C.c_uint64(0); h2d = C.c_uint64(0); d2h = C.c_uint64(0)
    sync_all()
    rc = lib.e2e_cold(h, int(op), compress, ptr(g0), n0, ptr(g1a), n1, int(args.e2e_steps + 1), ptr(ms), C.byref(cnt), C.byref(h2d), C.byref(d2h))
    assert rc == 0, "e2e_cold failed"
    assert cnt.value == total_bits, f"e2e (cold) result count {cnt.value} != device-resident run {total_bits}"
    cold_ms = float(np.mean(ms[1:]))                          # step 0 allocates the pinned ring and the result buffers
    a_ms, g_ms = C.c_double(0), C.c_double(0)
    rc = lib.e2e_cold_split(h, int(op), compress, ptr(g0), n0, ptr(g1a), n1, C.byref(a_ms), C.byref(g_ms))
    assert rc == 0
    # ---- warm: sources resident in a device_set ----
    wms = np.zeros(args.steps); wd2h = C.c_uint64(0)
    sync_all()
    rc = lib.e2e_warm(h, int(op), compress, ptr(g0), n0, ptr(g1a), n1, 3, int(args.steps), ptr(wms), C.byref(cnt), C.byref(wd2h))
    assert rc == 0, f"e2e_warm failed rc={rc}"
    assert cnt.value == total_bits, "e2e (warm) result differs from the device-resident run"
    warm_ms = float(np.mean(wms))
    # ---- result bvector vs the reference aggregator on the same bvectors (rank 0 only: single-threaded reference) ----
    chk = None
    if int(os.environ.get("RANK", "0")) == 0 and not args.no_e2e_check:
        eq = C.c_int(0); rcnt = C.c_uint64(0); rms = C.c_double(0)
        rc = lib.e2e_check(h, int(op), compress, ptr(g0), n0, ptr(g1a), n1, C.byref(eq), C.byref(rcnt), C.byref(rms))
        assert rc == 0
        chk = {"compare_eq_0_and_calc_stat_equal": bool(eq.value), "reference_count": int(rcnt.value), "reference_1thread_ms": rms.value}
        assert eq.value, "bm::b200::aggregator result differs from bm::aggregator on the same bvectors"
    lib.e2e_free(h)
    # ---- cold again, for applications that keep their bvectors on the page-locked slab allocator (bm::b200::slab_bvector,
    #      bitmagic_b200/include/bmb200_alloc.hpp): the slabs go up by DMA as they lie, the gather happens on the device ----
    slab = None
    es = E2E("libbmb200_e2e_slab.so")
    if world == 1 and es.ok() and not args.no_e2e_slab and mem_available_gb() >= need_gb:
        try:       # an optional leg: page-locking ~17 GB may be refused on a small box -- that must not take the line down
            ctx.trim()
            t0 = time.perf_counter()
            hs = build_bvectors(es.lib)
            build_s = time.perf_counter() - t0
            nsl, sbytes = C.c_uint64(0), C.c_uint64(0)
            es.lib.e2e_slab_info(C.byref(nsl), C.byref(sbytes))
            sms = np.zeros(args.e2e_steps + 2); scnt = C.c_uint64(0); sh2d = C.c_uint64(0); sd2h = C.c_uint64(0)
            rc = es.lib.e2e_cold(hs, int(op), compress, ptr(g0), n0, ptr(g1a), n1, int(args.e2e_steps + 2), ptr(sms), C.byref(scnt), C.byref(sh2d), C.byref(sd2h))
            assert rc == 0, "e2e_cold (slab allocator) failed"
            assert scnt.value == total_bits, f"e2e (cold, slab allocator) result count {scnt.value} != device-resident run {total_bits}"
            sa_ms, sg_ms = C.c_double(0), C.c_double(0)
            rc = es.lib.e2e_cold_split(hs, int(op), compress, ptr(g0), n0, ptr(g1a), n1, C.byref(sa_ms), C.byref(sg_ms))
            assert rc == 0
            seq = None
            if not args.no_e2e_check:
                eq = C.c_int(0); rcnt = C.c_uint64(0); rms = C.c_double(0)
                rc = es.lib.e2e_check(hs, int(op), compress, ptr(g0), n0, ptr(g1a), n1, C.byref(eq), C.byref(rcnt), C.byref(rms))
                assert rc == 0 and eq.value, "slab_bvector result differs from bm::aggregator on the same bvectors"
                seq = bool(eq.value)
            es.lib.e2e_free(hs)
            scold = float(np.mean(sms[2:]))        # step 0 allocates (result blocks come from the slab heap too: it grows once), step 1 re-sizes the device mirror for that
            slab = {"value": src_blocks_all / (scold * 1e-3), "unit": "blocks/s", "ms_per_step": scold, "host_slabs": int(nsl.value),
                    "h2d_bytes_per_step": int(sbytes.value) + 8 * dset.n_vec * dset.n_blocks, "h2d_gbs": sbytes.value / scold / 1e6,
                    "split_ms": {"device_set_assign(slab DMA | walk+layout, gather kernel)": sa_ms.value, "aggregate_on_resident(kernel+D2H+bvector)": sg_ms.value},
                    "pcie_floor_ms": sbytes.value / 55e9 * 1e3, "compare_eq_0_and_calc_stat_equal": seq, "bvector_build_s": build_s,
                    "path": "cold on bm::b200::slab_bvector: bmb200_host_slabs_prefetch + bmb200_set_upload_slabs (no host packing) + kernel + D2H + result bvector"}
            ctx.trim()
        except Exception as ex:                                   # (a result mismatch lands here too and is reported as such)
            slab = {"unavailable": f"{type(ex).__name__}: {ex}"}
    t = torch.tensor([cold_ms, warm_ms], dtype=torch.float64, device=f"cuda:{device}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    cold_ms, warm_ms = float(t[0].item()), float(t[1].item())
    # `value` = the WARM call: both arms then time the same thing -- one aggregator call with the operands already in the implementation's
    # own storage (the reference arm's bm::bvector<> objects are built once outside ITS timed region too), host bvector pointers in,
    # result bm::bvector<> out; per step the group member ids go H2D and the result comes back D2H.  `cold` is the same call with nothing
    # resident: it additionally pays, every step, for building the device copy (walk + pack + 13.5 GB over PCIe).
    return {"value": src_blocks_all / (warm_ms * 1e-3), "unit": "blocks/s", "ms_per_step": warm_ms,
            "h2d_bytes_per_step": 4 * (n0 + n1), "d2h_bytes_per_step": int(wd2h.value),
            "path": "warm: bm::b200::aggregator::combine_* on real bm::bvector<> sources that are resident in a bm::b200::device_set (uploaded once from "
                    "those bvectors, outside the timed region, like the reference arm's bvectors are built once); per step: member ids H2D, kernel, "
                    "result D2H, result bm::bvector<> materialised and compared with bm::aggregator's",
            "cold": {"value": src_blocks_all / (cold_ms * 1e-3), "unit": "blocks/s", "ms_per_step": cold_ms,
                     "h2d_bytes_per_step": int(h2d.value), "d2h_bytes_per_step": int(d2h.value), "h2d_gbs": h2d.value / cold_ms / 1e6,
                     "path": "cold: the same call with nothing resident (tree walk + layout + threaded pack + H2D + kernel + D2H + result bvector, every step)",
                     "split_ms": {"device_set_assign(walk+layout+pack+H2D)": a_ms.value, "aggregate_on_resident(kernel+D2H+bvector)": g_ms.value},
                     "pcie_floor_ms": h2d.value / 55e9 * 1e3, "slab_allocator": slab},
            "host_threads": thr, "numa_node": node.value, "check": chk}


DUMP_SAMPLE_COLS = 256


def dump_outputs(out_dir, bm, res, meta, total_bits):
    """float64 .npy files of the last timed step's result (exact: every value is an integer below 2^32)."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    kind, pop, dig, nr = meta
    cols = np.sort(np.random.default_rng(20261017).choice(kind.size, size=min(DUMP_SAMPLE_COLS, kind.size), replace=False))
    words = np.zeros((cols.size, 2048), np.float64)
    for i, c in enumerate(cols):
        k, bits, gap = res.fetch_column(int(c))
        bv = bm.BVector(1)
        if k == bm.BLK_BIT:
            bv.set_bits(0, bits)
        elif k == bm.BLK_GAP:
            bv.set_gap(0, gap)
        elif k == bm.BLK_FULL:
            bv.set_full(0)
        words[i] = bv.block_words(0)
    arrays = {"kind": kind, "popcnt": pop, "digest_lo": dig & np.uint64(0xFFFFFFFF), "digest_hi": dig >> np.uint64(32), "gap_runs": nr,
              "total_bits": np.array([total_bits], np.uint64), "sample_cols": cols, "sample_words": words}
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", np.asarray(a).astype(np.float64))


class _StdoutToStderr:
    """Everything libraries print while the bench runs (NCCL's version banner, warnings ...) goes to stderr, so that stdout
    carries exactly ONE line: the JSON result."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)
        return False


def main():
    with _StdoutToStderr():
        line = _main()
    if line is not None:
        print(json.dumps(line), flush=True)


def timed_resident(args, bm, torch, ctx, dset, op, g0, g1, flags, world, dist, dev, stream, n_cols, rank, sample_clocks=True):
    """W warm-up + K timed steps of the device-resident aggregation (+ the library's own exchange when world > 1)."""
    res = bm.aggregate(ctx, dset, op, g0, g1, flags)     # allocates the result buffers once
    ctx.sync()

    # diagnostic switch (the N>1 line always runs the exchange): BENCH_SELF_EXCHANGE=1 runs the exchange machinery on ONE GPU with a
    # 1-rank communicator, to separate its stream-level cost from what the peers add
    exchange = world > 1 or bool(os.environ.get("BENCH_SELF_EXCHANGE"))

    def step():
        bm.aggregate(ctx, dset, op, g0, g1, flags, result=res)
        if exchange:
            ctx.exchange_popcounts(res)                  # side stream: overlaps the next step's kernel

    l0 = ctx.launch_count()
    for _ in range(args.warmup):
        step()
    if exchange:
        ctx.exchange_fence()
    torch.cuda.synchronize(dev)
    launches_per_step = (ctx.launch_count() - l0) // args.warmup

    sampler = ClockSampler(dev.index) if (rank == 0 and sample_clocks) else None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    if sampler:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # a dedicated event pair around the dominant kernel of every step (aggregate launch only)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    if world > 1:
        # the host-side barrier above releases the ranks' CPU threads up to a millisecond apart, and with a per-step exchange a rank
        # that starts late is waited for by all others (measured: 0.7 ms of start skew = 37 us on each of 20 steps).  A device-side
        # rendezvous right in front of the first event makes every rank's timed region start together on the GPUs.
        sync_t = torch.zeros(1, device=dev)
        dist.all_reduce(sync_t)
    ev0.record(stream)
    for i in range(args.steps):
        kev[i][0].record(stream)
        bm.aggregate(ctx, dset, op, g0, g1, flags, result=res)
        kev[i][1].record(stream)
        if exchange:
            ctx.exchange_popcounts(res)
    if exchange:
        ctx.exchange_fence()                             # the launching stream waits for every exchange: they are inside the timed region
    ev1.record(stream)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    total_ms = ev0.elapsed_time(ev1)
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return res, float(t.item()) / args.steps, kern_ms, clocks, launches_per_step


def _main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=list(WORKLOADS))
    ap.add_argument("--cols", type=int, default=0, help="override block columns per GPU (reduced runs are flagged)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-e2e-check", action="store_true")
    ap.add_argument("--no-e2e-slab", action="store_true", help="skip the cold e2e leg on slab-allocator bvectors (N=1 only; page-locks ~ the set size)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the extra config-5 shard line that 8-GPU runs carry")
    ap.add_argument("--cpu-cols", type=int, default=256, help="block columns in the 1-thread cpu_baseline sample")
    ap.add_argument("--ref-threads", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result arrays to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        return run_reference(args)

    import torch
    import bitmagic_b200 as bm

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = torch.device(f"cuda:{local}")

    w = WORKLOADS[args.workload]
    n_cols = args.cols or w["n_blocks"]
    ctx = bm.Context(local)
    all_cpus = os.sched_getaffinity(0)
    numa_node = ctx.bind_host_numa()          # host threads + pinned staging next to this GPU's PCIe root (GPUs 0-3 / 4-7 sit on different nodes)
    gpu_cpus = os.sched_getaffinity(0)
    stream = torch.cuda.current_stream(dev)
    ctx.set_stream(stream.cuda_stream)
    exchange = None
    if world == 1 and os.environ.get("BENCH_SELF_EXCHANGE"):
        ctx.comm_init(1, 0, bytes(ctx.comm_unique_id()))
    if world > 1:
        # the library's own communicator: rank 0 makes the id, torch.distributed only ships its 128 bytes
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(ctx.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        ctx.comm_init(world, rank, bytes(idt.cpu().numpy().tobytes()))
        exchange = "bmb200_exchange_popcounts: one ncclAllGather of (columns + 2) u32 per rank on a side stream, step i's exchange overlaps step i+1's kernel; the last one is fenced inside the timed region"

    dens, seed, optimize = workload_inputs(args.workload, rank)
    op, g0, g1, flags = workload_groups(args.workload)
    t0 = time.time()
    dset = bm.DeviceSet.synth(ctx, w["n_vec"], n_cols, dens, seed, optimize)
    ctx.sync()
    t_synth = time.time() - t0
    counts, gap_words = device_set_stats(ctx, dset, torch)
    n_src_blocks = counts["bit"] + counts["gap"] + counts["full"]

    res, ms_per_step, kern_ms, clocks, launches_per_step = timed_resident(args, bm, torch, ctx, dset, op, g0, g1, flags, world, dist, dev, stream, n_cols, rank)

    total_bits, any_ = res.total()
    kind_r, pop_r, dig_r, nr_r = res.meta()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, bm, res, (kind_r, pop_r, dig_r, nr_r), total_bits)
    res_bytes = int((kind_r == bm.BLK_BIT).sum()) * 8192 + int(2 * (nr_r[kind_r == bm.BLK_GAP].astype(np.int64) + 1).sum())
    # algorithmic bytes (SURVEY 8d): stored source bytes (bit 8192 B, GAP 2*(len+1) B) + result blocks written + 12 B meta per column
    alg_bytes = counts["bit"] * 8192 + gap_words * 2 + res_bytes + n_cols * 12
    xchg = None
    if world > 1:
        gtot, rtot, gpop = ctx.exchange_fetch(world, n_cols, want_popcounts=True)
        assert int(rtot[rank]) == int(total_bits), "exchange: this rank's cardinality did not come back"
        assert np.array_equal(gpop[rank], pop_r), "exchange: this rank's per-column popcounts did not come back"
        tb = torch.tensor([int(total_bits)], dtype=torch.int64, device=dev)
        dist.all_reduce(tb)                                  # the same sum over torch.distributed's own NCCL communicator
        assert int(tb.item()) == int(gtot) == int(gpop.astype(np.int64).sum()), "exchange: global cardinality differs from an all_reduce of the rank totals"
        mode = ctx.exchange_mode()
        exchange = {2: "bmb200_exchange_popcounts over peer memory: every rank's exchange buffer is mapped by all ranks (CUDA IPC); a small kernel behind the "
                       "aggregation kernel stores this rank's (columns + 2) u32 row into every peer over NVLink and publishes a sequence number; "
                       "the last exchange is awaited inside the timed region",
                    1: "bmb200_exchange_popcounts: one ncclAllGather of (columns + 2) u32 per rank on a side stream, step i's exchange overlaps step "
                       "i+1's kernel; the last one is fenced inside the timed region"}.get(mode, exchange)
        xchg = {"global_result_bits": int(gtot), "collective": exchange, "mode": mode, "checked": "own row + all_reduce of the rank totals"}

    src_blocks_all = torch.tensor([n_src_blocks], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(src_blocks_all)
    src_blocks_all = float(src_blocks_all.item())
    value = src_blocks_all / (ms_per_step * 1e-3)

    # ---- parity: every column against the reference on the host (rank 0; its own shard) ----
    parity = None
    cpu = None
    if rank == 0 and not args.no_parity:
        need = 2.3 * dset.stored_bytes() / 2**30
        if mem_available_gb() > need + 8:
            os.sched_setaffinity(0, all_cpus)     # the reference gets every core of the box, not only this GPU's NUMA node
            parity, host_src_blocks, host_stored = full_parity(args.workload, n_cols, rank, (kind_r, pop_r, dig_r, nr_r), os.cpu_count() or 1)
            parity["ranks_checked"] = [0]
            parity["inputs_equal"] = bool(host_src_blocks == n_src_blocks and host_stored == dset.stored_bytes())
            os.sched_setaffinity(0, gpu_cpus)
            assert parity["equal"] and parity["inputs_equal"], f"PARITY FAILURE against the reference: {parity}"
        else:
            parity = {"skipped": f"host memory {mem_available_gb():.0f} GB < {need + 8:.0f} GB"}

    # ---- e2e: real bvectors through the C++ binding ----
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, ctx, dset, local, world, dist, torch, op, g0, g1, flags, total_bits, src_blocks_all)

    # ---- CPU baseline rows (rank 0): 1 thread on a bounded sample; all cores = the parity run above (whole workload) ----
    if rank == 0 and world == 1 and not args.no_cpu:
        import orclib
        ncs = min(args.cpu_cols, n_cols)
        ps_s = dset.download(0, ncs)
        src_s = int((ps_s.kinds() != 0).sum())
        os.sched_setaffinity(0, all_cpus)
        if orclib.have_ref():
            job = orclib.RefJob(ps_s, op, g0, g1, flags, threads=1)
            job.run(1)
            sec, tot = job.run(3)
            sec = float(np.min(sec)); job.free()
            kind_c, simd = "reference", orclib.ref().ref_simd().decode()
        else:
            t0 = time.perf_counter(); o = orclib.oracle_aggregate(ps_s, op, g0, g1, flags); sec = time.perf_counter() - t0
            tot = int(o[1].sum()); kind_c, simd = "port", "scalar"
        assert tot == int(pop_r[:ncs].sum()), "CPU baseline and GPU disagree on the sampled columns"
        cpu = {"value": src_s / sec, "unit": "blocks/s", "cores": 1, "kind": kind_c, "simd": simd, "nproc": os.cpu_count(), "cpu": cpu_model(),
               "sample": f"first {ncs} of {n_cols} block columns x {w['n_vec']} vectors ({ps_s.stored_bytes() / 2**20:.0f} MiB), {sec * 1e3:.0f} ms, bvectors built before the clock starts",
               "gbs": ps_s.stored_bytes() / sec / 1e9, "checked_equal_popcount": True}
        if parity and "ref_ms" in parity:
            cpu["all_cores"] = {"value": n_src_blocks / (parity["ref_ms"] * 1e-3), "unit": "blocks/s", "cores": parity["ref_threads"],
                                "ms": parity["ref_ms"], "sample": "the whole workload (the parity run)"}

    # ---- config 5 rides along on 8-GPU runs: each rank's shard IS configs[4] (4096 x 2^32 bits over 8 GPUs) ----
    c5 = None
    if world == int(os.environ.get("BENCH_C5_WORLD", "8")) and args.workload == "c3" and not args.no_c5:      # (the env override lets a 2-GPU box exercise this path)
        dset.free(); res.free()
        w5 = WORKLOADS["c5"]
        d5, s5, o5 = workload_inputs("c5", rank)
        op5, g05, g15, f5 = workload_groups("c5")
        ds5 = bm.DeviceSet.synth(ctx, w5["n_vec"], w5["n_blocks"], d5, s5, o5)
        ctx.sync()
        cnt5, gw5 = device_set_stats(ctx, ds5, torch)
        a5 = argparse.Namespace(**vars(args)); a5.steps = min(args.steps, 10)
        r5, ms5, k5, _, _ = timed_resident(a5, bm, torch, ctx, ds5, op5, g05, g15, f5, world, dist, dev, stream, w5["n_blocks"], rank, sample_clocks=False)
        kk, pp, dd, nn = r5.meta()
        rb5 = int((kk == bm.BLK_BIT).sum()) * 8192 + int(2 * (nn[kk == bm.BLK_GAP].astype(np.int64) + 1).sum())
        alg5 = cnt5["bit"] * 8192 + gw5 * 2 + rb5 + w5["n_blocks"] * 12
        nb5 = torch.tensor([cnt5["bit"] + cnt5["gap"] + cnt5["full"]], dtype=torch.int64, device=dev)
        dist.all_reduce(nb5)
        g5, _, _ = ctx.exchange_fetch(world, w5["n_blocks"], want_popcounts=False)
        peak, _ = measured_peak_gbs()
        c5 = {"workload": "c5: " + w5["desc"], "n_gpus": world, "steps": a5.steps, "ms_per_step": ms5, "value": float(nb5.item()) / (ms5 * 1e-3), "unit": "blocks/s",
              "kernel_ms": k5, "algorithmic_bytes_per_gpu": int(alg5), "gbs_per_gpu": alg5 / (k5 * 1e-3) / 1e9, "frac_of_peak": alg5 / (k5 * 1e-3) / 1e9 / peak,
              "global_result_bits": int(g5)}
        r5.free(); ds5.free()

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
        reduced = bool(args.cols and args.cols != w["n_blocks"])
        traffic, traffic_src = (None, None) if reduced else profiled_traffic(args.workload)
        line = {
            "metric": "aggregator input 64Kbit-blocks/s", "value": value, "unit": "blocks/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": args.workload + ": " + w["desc"], "n_vec": w["n_vec"], "block_columns_per_gpu": n_cols,
                       "reduced": reduced,
                       "l2": f"inputs ({alg_bytes / 2**30:.2f} GiB per GPU) larger than the 126 MB L2; no flush needed",
                       "parallelism": f"block-range sharded x{world}", "source_blocks": counts, "synth_s": round(t_synth, 2),
                       "exchange": exchange, "numa_node": numa_node},
            "gbs_per_gpu": alg_bytes / (ms_per_step * 1e-3) / 1e9,
            "clocks": clocks, "gpu_launches": int(launches_per_step * args.steps),
            "e2e": e2e,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "agg_kernel<%s>" % w["op"], "kernel_ms": kern_ms,
                         "algorithmic_bytes_per_launch": int(alg_bytes), "peak_source": peak_src},
            "cpu_baseline": cpu,
            "parity": parity,
            "result_bits": int(total_bits),
        }
        if xchg:
            line["exchange"] = xchg
        if c5:
            line["c5"] = c5
    else:
        line = None
    if world > 1:
        ctx.comm_destroy()
        dist.destroy_process_group()
    return line


if __name__ == "__main__":
    main()
