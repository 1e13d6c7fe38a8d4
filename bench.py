#!/usr/bin/env python3
"""bench.py -- rows scanned/s of the LogsQL block-scan hot path on B200 (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # GPU arm (libvlscan.so)
    python bench.py --impl reference [--gpus N] [--steps K] ...    # reference arm: the CPU algorithm on the host cores
    python bench.py ... --dump-outputs DIR                         # also write what the last timed step computed to DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic blocks:  bm.init/setBits + filter.applyToBlockSearch for every
block (lib/logstorage/block_search.go:207-215).

Workload at N=1: BASELINE.json configs[2] (C3, the config the north-star target is quoted on and the largest one that fits one GPU):
`_msg:~"conn.*refused"` over 1 B vlogsgenerator-shaped rows, 32 fields => 2000 rows/block by the 2 MB rule, 500 000 blocks, ~142 GB
of `_msg` bytes + lens items + bloom filters resident in HBM when the timed region starts (`value`).  `e2e` is the same filter through
the C-ABI call vlscan_scan_batch on pinned HOST buffers holding the blocks in their on-disk form (ZSTD frames), H2D + device decode +
scan + D2H inside the timed region, on the first --e2e-rows rows of the same data set per step (a search worker hands the part over
batch by batch; host staging of all 1e9 rows would need ~60 GB of pinned memory and minutes of writer-side compression).
C2 and C4 (BASELINE.json configs[1], configs[3]) are measured in the same run and reported under `extra_workloads`.

Parity inside the bench: the first --cpu-sample-rows rows of the benched batch are also scanned by the CPU oracle; the digest of its
bitmaps (xor of XXH64(block bitmap) * (2 * block + 1)) must equal the digest the device computes over the same blocks of the timed
scan's result (`parity`), and the end-to-end leg must reproduce the resident leg's bitmaps digest and match count.

N>1: every rank scans its own shard of an N x larger data set (blocks are independent: weak scaling, no data-path collective); the
ranks accumulate {rows, rows_matched, blocks_matched, values_bytes} on the device and all-reduce them over NCCL ONCE, after the last
step, inside the timed region (SURVEY 8e).

The reference (Go) cannot run here (no Go toolchain); the reference arm / cpu_baseline time the oracle's restatement of the same
per-block algorithm (kind "port"; linked against the reference's own libzstd 1.5.7 when oracle/_ref was built) on all host cores,
on a bounded sample of the same workload.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20250718
WORKLOADS = {
    # name: rows per rank, fields, rows/block, columns_mask, filter builder, logsql
    "C1": dict(rows=1_000_000, fields=8, rows_per_block=6400, mask=0b0001, logsql='_msg:"error"', tree=lambda F: F.phrase("_msg", "error")),
    "C2": dict(rows=100_000_000, fields=16, rows_per_block=3000, mask=0b0011, logsql='_msg:"timeout" AND level:error',
               tree=lambda F: F.and_([F.phrase("_msg", "timeout"), F.phrase("level", "error")])),
    "C3": dict(rows=1_000_000_000, fields=32, rows_per_block=2000, mask=0b0001, logsql='_msg:~"conn.*refused"', tree=lambda F: F.regexp("_msg", "conn.*refused")),
    "C4": dict(rows=125_000_000, fields=32, rows_per_block=2000, mask=0b1101, logsql='_msg:"GET" AND path:api* AND status:in(500,502,503)',
               tree=lambda F: F.and_([F.phrase("_msg", "GET"), F.prefix("path", "api"), F.in_("status", ["500", "502", "503"])])),
}
METRIC = "log rows scanned/sec (LogsQL phrase+regex)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="vlscan", choices=["vlscan", "reference"])
    ap.add_argument("--workload", default="C3", choices=sorted(WORKLOADS))
    ap.add_argument("--rows", type=int, default=0, help="rows per rank (default: the workload's)")
    ap.add_argument("--hot-block-permille", type=int, default=1000, help="block clustering knob: fraction of blocks holding vocabulary rows")
    ap.add_argument("--hit-row-permille", type=int, default=60, help="selectivity knob: vocabulary rows inside hot blocks")
    ap.add_argument("--vocab-focus", type=int, default=0, help="1..12: every vocabulary row carries that vocabulary entry (selectivity studies); 0: uniform draw, the headline setting")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-rows", type=int, default=100_000_000, help="rows per end-to-end step (the first rows of the rank's shard)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-stage", default="ondisk", choices=["ondisk", "decoded"], help="form of the host blocks handed to vlscan_scan_batch")
    ap.add_argument("--cpu-sample-rows", type=int, default=12_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra workloads (C2, C4) measured next to the headline at N=1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (rank 0's shard) as DIR/<name>.npy, "
                    "so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "vlscan":
        ap.error("--dump-outputs writes the device scan's outputs: --impl vlscan only")
    return args


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "samples": len(sm), "reasons": reasons}


def hbm_peak():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def ncu_traffic(workload, rows):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu --set full capture of this launch size"""
    try:
        for rec in json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic_r02.json"))):
            if rec["workload"] == workload and int(rec["rows"]) == int(rows):
                return rec
    except Exception:
        pass
    return None


def host_info():
    info = {"cores": os.cpu_count() or 1}
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                info["cpu_model"] = line.split(":", 1)[1].strip()
                break
        info["loadavg_1m"] = float(open("/proc/loadavg").read().split()[0])
    except Exception:
        pass
    return info


def bind_to_gpu_numa_node(local_rank):
    """N > 1: the ranks of a box share its host cores, its memory controllers and its PCIe roots.  Keep a rank's threads (and with them the
    pinned staging memory they touch first) on the NUMA node its GPU hangs off, so that H2D copies do not cross the socket interconnect."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception:
        return None


def oracle():
    ref = os.path.join(ROOT, "oracle", "_ref", "liboracle_zstd157.so")
    if os.path.exists(ref):
        os.environ.setdefault("VLORACLE_LIB", ref)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vloracle
    return vloracle, ("reference libzstd 1.5.7 (oracle/_ref)" if os.environ.get("VLORACLE_LIB") == ref else "system libzstd")


def cpu_port(wl, gen_kw, sample_rows, threads, target_secs=10.0, post_zstd=False, block_lo=0):
    """The reference's per-block algorithm restated on the CPU (oracle/), all host threads pinned, bounded sample. -> rows/s, info"""
    vloracle, zlib = oracle()
    cfg = vloracle.GenConfig(**gen_kw)
    total_blocks = (gen_kw["total_rows"] + wl["rows_per_block"] - 1) // wl["rows_per_block"]
    nb = max(1, min(sample_rows // wl["rows_per_block"], total_blocks - block_lo))
    flt = wl["tree"](vloracle.Filter)
    # calibrate the number of passes so that the timed region holds ~target_secs of CPU work (bounded sample, repeated)
    r = vloracle.scan_generated(cfg, flt, block_lo, block_lo + nb, threads, post_zstd=post_zstd, pin=True)
    first = r
    passes = int(max(1, min(400, target_secs / max(r["secs"], 1e-4))))
    if passes > 1:
        r = vloracle.scan_generated(cfg, flt, block_lo, block_lo + nb, threads, passes=passes, post_zstd=post_zstd, pin=True)
    rows = int(r["stats"][1])
    rate = rows * passes / r["secs"]
    return rate, dict(rows=rows, blocks=nb, secs=r["secs"], passes=passes, matches=int(first["matches"]), digest=int(first["digest"]), values_bytes=int(r["stats"][3]), zstd=zlib)


def run_reference(args, wl, gen_kw, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    rates, info = [], None
    n = args.warmup + args.steps
    for i in range(n):
        rate, info = cpu_port(wl, gen_kw, args.cpu_sample_rows, threads, target_secs=min(8.0, 160.0 / n))
        if i >= args.warmup:
            rates.append(rate)
    value = statistics.median(rates)
    hi = host_info()
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": len(rates),
        "warmup": args.warmup, "ms_per_step": 1000.0 * info["rows"] * info["passes"] / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic (deterministic vlogsgenerator-shaped rows, seed %d)" % SEED,
        "config": {"workload": "%s: %s" % (args.workload, wl["logsql"]), "rows_per_step": info["rows"] * info["passes"], "rows_per_block": wl["rows_per_block"], "fields": wl["fields"],
                   "hot_block_permille": gen_kw["hot_block_permille"], "hit_row_permille": gen_kw["hit_row_permille"],
                   "note": "Go toolchain absent: the reference's per-block algorithm restated in C++ (oracle/), ZSTD-compressed values blocks included (%s), all host threads, pinned" % info["zstd"]},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port", "variant": "with-zstd", "spread": [min(rates), max(rates)], "cpu_model": hi.get("cpu_model"), "loadavg_1m": hi.get("loadavg_1m"),
                         "sample": "%d rows (%d blocks) of the %s workload x %d passes per step, median of %d steps" % (info["rows"], info["blocks"], args.workload, info["passes"], len(rates))},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def words_digest(vloracle, words, rows_list, key_base):
    """the oracle's digest formula over host bitmaps (vlo_scan_generated): xor of XXH64(block words) * (2 * key + 1) mod 2^64"""
    d, off = 0, 0
    for i, r in enumerate(rows_list):
        nw = (r + 63) // 64
        d ^= (vloracle.xxh64(words[off:off + nw].tobytes()) * (2 * (key_base + i) + 1)) & 0xFFFFFFFFFFFFFFFF
        off += nw
    return d


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, words, counts, block_rows):
    """What a caller of the resident scan receives, as float arrays of at most DUMP_BYTES in all: the match count of every block
    (block_match_counts), and the per-row match bits (0 / 1, block after block) of a fixed, seeded sample of the blocks (sample_match_bits)
    whose indices are sample_blocks - every block when the bitmaps fit.  The bits of a block are its bitmap words, least significant first."""
    import numpy as np
    nb = len(block_rows)
    word_off = np.concatenate(([0], np.cumsum((block_rows + 63) // 64)))
    k = min(nb, (DUMP_BYTES - 8 * nb - 4096) // (4 * int(block_rows.max()) + 8))
    pick = np.sort(np.random.default_rng(SEED).choice(nb, size=k, replace=False))
    bits = [np.unpackbits(words[word_off[b]:word_off[b + 1]].view(np.uint8), bitorder="little")[:block_rows[b]] for b in pick]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "block_match_counts.npy"), counts.astype(np.float64))
    np.save(os.path.join(out_dir, "sample_blocks.npy"), pick.astype(np.float64))
    np.save(os.path.join(out_dir, "sample_match_bits.npy"), np.concatenate(bits).astype(np.float32))


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = WORKLOADS[args.workload]

    def gen_args(w, rows):
        rows -= rows % w["rows_per_block"] if rows % w["rows_per_block"] and rows % w["rows_per_block"] < 64 else 0
        nb = (rows + w["rows_per_block"] - 1) // w["rows_per_block"]
        kw = dict(seed=SEED, total_rows=rows * world, rows_per_block=w["rows_per_block"], hot_block_permille=args.hot_block_permille,
                  hit_row_permille=args.hit_row_permille, columns_mask=w["mask"] | (args.vocab_focus << 8))
        if rows % w["rows_per_block"]:
            kw["total_rows"] = nb * w["rows_per_block"] * (world - 1) + rows if world > 1 else rows
        return rows, nb, kw

    rows, nb, gen_kw = gen_args(wl, args.rows or wl["rows"])
    if args.impl == "reference":
        run_reference(args, wl, gen_kw, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from victorialogs_b200 import scan as vs, shard

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libvlscan has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = vs.Ctx(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream, device=local_rank)
    peak, peak_src = hbm_peak()

    class _Arr:   # zero-copy torch view of the library's 4 x u64 totals vector
        def __init__(self, ptr):
            self.__cuda_array_interface__ = {"shape": (4,), "typestr": "<i8", "data": (ptr, False), "version": 2}

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    def measure(w, w_rows, w_nb, w_kw, steps, warmup, sample_clocks, capture=False):
        """resident scan of one workload -> dict; the batch stays alive in the returned dict until the caller frees it.
        capture: also return the bitmap words and match counts of the last timed step (`outputs`)"""
        gcfg = vs.GenConfig(**w_kw)
        block_lo = rank * w_nb
        t_gen = time.time()
        batch = ctx.generate(gcfg, block_lo, block_lo + w_nb)
        ctx.sync()
        t_gen = time.time() - t_gen
        prog = vs.Program(w["tree"](vs.Filter))
        acc = torch.zeros(4, dtype=torch.int64, device="cuda")

        def step():
            ctx.scan_resident(prog, batch, want_stats=False)
            if world > 1:   # the match counters of every step are summed on the device, on the scan's stream
                _, _, totals = ctx.result_device_ptrs()
                with torch.cuda.stream(stream):
                    acc.add_(torch.as_tensor(_Arr(totals), device="cuda"))

        for _ in range(max(warmup, 3)):
            step()
        sync_all()
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        acc.zero_()
        sync_all()
        ev0.record(stream)
        for _ in range(steps):
            step()
        if world > 1:
            with torch.cuda.stream(stream):
                shard.reduce_counters(acc)     # the only collective of the path: ONE final NCCL reduce of the match counters
        ev1.record(stream)
        sync_all()
        outputs = ctx.fetch(batch) if capture else None   # before any untimed scan below replaces the result
        clocks = None
        if sampler:
            # the timed region may be shorter than a few nvidia-smi sampling periods: keep the same load running (untimed) until the sampler
            # has seen ~1 s of it, so that `clocks` really is the SM clock / throttle state under this workload
            t_hold = time.perf_counter()
            while time.perf_counter() - t_hold < 1.0:
                ctx.scan_resident(prog, batch, want_stats=False)
                ctx.sync()
            clocks = sampler.stop()
        ms = ev0.elapsed_time(ev1)
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        # roofline of the dominant kernel (k_substr_scan): algorithmic bytes / its CUDA-event duration, averaged over fresh scans
        kms, kbytes, gms = [], 0, []
        for _ in range(min(steps, 10)):
            ctx.scan_resident(prog, batch, want_stats=False)
            s = ctx.last_scan_stats()
            kms.append(s.scan_kernel_ms)
            gms.append(s.gpu_ms)
            kbytes = s.scan_kernel_bytes
        st = ctx.last_scan_stats()
        k_avg = statistics.mean(kms) if kms else 0.0
        achieved = (kbytes / 1e9) / (k_avg / 1e3) if k_avg > 0 else 0.0
        step_bytes = st.values_bytes + st.bloom_probe_bytes + st.bitmap_bytes
        return dict(batch=batch, prog=prog, gcfg=gcfg, block_lo=block_lo, ms=ms, steps=steps, st=st, clocks=clocks, t_gen=t_gen, k_avg=k_avg, kbytes=kbytes, achieved=achieved,
                    step_bytes=step_bytes, share=(k_avg / statistics.mean(gms)) if gms and statistics.mean(gms) > 0 else None,
                    totals=acc.cpu().tolist() if world > 1 else None, outputs=outputs)

    # ---- the headline workload, resident -----------------------------------------------------------------------------------------
    fallback_note = None
    m = None
    want_rows = rows
    for attempt in range(4):
        try:
            m = measure(wl, rows, nb, gen_kw, args.steps, args.warmup, True, capture=bool(args.dump_outputs) and rank == 0)
            break
        except vs.VlscanError as e:   # does not fit this GPU next to whatever else lives on it: fall back to the largest row count that does
            # (not when dumping: a dump must hold the outputs of the inputs the arguments name, or two dumps could not be compared)
            if "memory" not in str(e).lower() or attempt == 3 or args.dump_outputs:
                raise
            fallback_note = "%d rows/GPU did not fit (%s)" % (rows, str(e)[:80])
            rows, nb, gen_kw = gen_args(wl, int(rows * 0.8))
    if m["outputs"] is not None:
        first = m["block_lo"] * wl["rows_per_block"]
        block_rows = np.minimum(wl["rows_per_block"], gen_kw["total_rows"] - first - wl["rows_per_block"] * np.arange(nb, dtype=np.int64))
        dump_outputs(args.dump_outputs, *m["outputs"], block_rows)
        m["outputs"] = None
    st, batch, prog = m["st"], m["batch"], m["prog"]
    device_bytes = batch.device_bytes
    _, resident_counts = ctx.fetch(batch, bitmaps=False, counts=True)

    # ---- parity of the benched scan against the CPU oracle on its first blocks (device digest vs oracle digest) + CPU baselines ----
    cpu, cpu_post, parity = None, None, None
    pblocks = max(1, min(args.cpu_sample_rows // wl["rows_per_block"], nb))
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        hi = host_info()
        rate, info = cpu_port(wl, gen_kw, args.cpu_sample_rows, threads)
        dev_digest = ctx.result_digest(0, info["blocks"], m["block_lo"])
        dev_matches = int(resident_counts[:info["blocks"]].sum()) if resident_counts is not None else None
        parity = {"checked_rows": info["rows"], "checked_blocks": info["blocks"], "digest_device": "%016x" % dev_digest, "digest_oracle": "%016x" % info["digest"],
                  "matches_device": dev_matches, "matches_oracle": info["matches"], "ok": dev_digest == info["digest"] and (dev_matches is None or dev_matches == info["matches"]),
                  "how": "xor over blocks of XXH64(bitmap words) * (2 * block + 1): vlscan_result_digest on the result of the timed resident scan vs the CPU oracle on the same generated blocks"}
        cpu = {"value": rate, "unit": "rows/s", "cores": threads, "kind": "port", "variant": "with-zstd", "cpu_model": hi.get("cpu_model"), "loadavg_1m": hi.get("loadavg_1m"), "zstd": info["zstd"],
               "sample": "first %d rows (%d blocks) of the %s workload x %d passes, ZSTD-compressed values blocks, %d pinned threads, %.2f s" % (info["rows"], info["blocks"], args.workload, info["passes"], threads, info["secs"])}
        rate2, info2 = cpu_port(wl, gen_kw, args.cpu_sample_rows, threads, target_secs=5.0, post_zstd=True)
        cpu_post = {"value": rate2, "unit": "rows/s", "cores": threads, "kind": "port", "variant": "post-zstd",
                    "sample": "same blocks, values blocks decompressed before the timed region (the input stage of the resident scan), %d passes, %.2f s" % (info2["passes"], info2["secs"])}

    batch.free()
    m["batch"] = None

    # ---- end to end through the C ABI on pinned host buffers ------------------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        try:
            e_nb = max(1, min(nb, args.e2e_rows // wl["rows_per_block"]))
            e_rows = min(rows, e_nb * wl["rows_per_block"])
            sub = ctx.generate(m["gcfg"], m["block_lo"], m["block_lo"] + e_nb)
            ctx.scan_resident(prog, sub, want_stats=False)
            sub_digest = ctx.result_digest(0, e_nb, m["block_lo"])
            sub_matched = int(ctx.last_scan_stats().rows_matched)
            host = ctx.download(sub)
            sub.free()
            t_comp = 0.0
            if args.e2e_stage == "ondisk":
                # the reference's writer re-encodes every values block into its on-disk form (ZSTD frames); the scan call then ships the
                # compressed bytes and regenerates them on the device.  Not timed: it is the ingestion side.
                t1 = time.perf_counter()
                disk = host.compress(threads=max(1, (os.cpu_count() or 1) // world))   # ranks share the host cores
                t_comp = time.perf_counter() - t1
                del host
                host = disk
            # host threads the library may use inside an upload (ZSTD header walk); the ranks of a box share its cores
            os.environ.setdefault("VLSCAN_HOST_THREADS", str(max(1, min(32, (os.cpu_count() or 1) // world))))
            nwords = sum((r + 63) // 64 for r in host.rows)
            words = np.zeros(max(nwords, 1), dtype=np.uint64)
            counts = np.zeros(max(host.nblocks, 1), dtype=np.uint32)
            ctx.scan_batch(prog, host, words, counts)   # warm-up (allocations)
            sync_all()
            t0 = time.perf_counter()
            est = None
            for _ in range(args.e2e_steps):
                _, _, est = ctx.scan_batch(prog, host, words, counts)
            sync_all()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
            vloracle, _ = oracle()
            host_digest = words_digest(vloracle, words, list(host.rows), m["block_lo"]) if rank == 0 else None
            e2e = {"value": e_rows * world * args.e2e_steps / dt, "unit": "rows/s", "h2d_bytes_per_step": int(est.h2d_bytes) * world, "d2h_bytes_per_step": int(est.d2h_bytes) * world,
                   "ms_per_step": 1000 * dt / args.e2e_steps, "steps": args.e2e_steps, "rows_per_step_per_gpu": e_rows, "matched": int(counts.sum()),
                   "input_stage": "on-disk values blocks (ZSTD frames, decoded on the device)" if args.e2e_stage == "ondisk" else "decoded values blocks",
                   "host_bytes": int(host.bytes), "writer_compress_seconds": round(t_comp, 2), "host_threads": int(os.environ["VLSCAN_HOST_THREADS"]),
                   "matched_equals_resident": int(counts.sum()) == sub_matched,
                   "digest_equals_resident": (host_digest == sub_digest) if host_digest is not None else None,
                   "note": "each step = one vlscan_scan_batch over the first %d rows of the rank's shard (a search worker submits a part batch by batch)" % e_rows}
            del host
        except Exception as e:   # pinned host memory for the batch may not be available
            e2e = {"value": None, "unit": "rows/s", "error": str(e)[:200]}

    # ---- the other single-GPU configs of BASELINE.json, same run -------------------------------------------------------------------------
    extra = {}
    if not args.no_extra:
        # N > 1: C4 is BASELINE.json configs[3] - "1B rows block-sharded 8xB200" is 125 M rows per GPU, so at N = 8 this IS that configuration
        for name in (("C2", "C4") if world == 1 else ("C4",)):
            if name == args.workload:
                continue
            try:
                w = WORKLOADS[name]
                w_rows, w_nb, w_kw = gen_args(w, w["rows"])
                x = measure(w, w_rows, w_nb, w_kw, 10, 3, False)
                extra[name] = {"workload": "%s: %s over %d rows/GPU x %d GPU(s), %d fields" % (name, w["logsql"], w_rows, world, w["fields"]), "value": w_rows * world * x["steps"] / (x["ms"] / 1e3), "unit": "rows/s",
                               "ms_per_step": x["ms"] / x["steps"], "rows_matched": int(x["st"].rows_matched), "gpu_launches_per_step": int(x["st"].gpu_launches),
                               "step_hbm_gbs_per_gpu": (x["step_bytes"] / 1e9) / (x["ms"] / x["steps"] / 1e3),
                               "roofline": {"kernel": "k_substr_scan", "achieved": x["achieved"], "peak": peak, "unit": "GB/s", "frac": x["achieved"] / peak, "kernel_ms_per_launch": x["k_avg"],
                                            "algorithmic_bytes_per_launch": int(x["kbytes"]), "kernel_share_of_step": x["share"]}}
                x["batch"].free()
            except Exception as e:
                extra[name] = {"error": str(e)[:200]}

    # ---- bloom-first staging on clustered data: C2 with vocabulary rows in 1 block of 10 (the bloom filters rule the others out) ----------------
    bloom_first = None
    if world == 1 and not args.no_extra and not args.no_e2e:
        try:
            w = WORKLOADS["C2"]
            b_rows, b_nb, b_kw = gen_args(w, min(w["rows"], args.e2e_rows))
            b_kw["hot_block_permille"] = 100
            sub = ctx.generate(vs.GenConfig(**b_kw), 0, b_nb)
            host = ctx.download(sub)
            sub.free()
            disk = host.compress(threads=os.cpu_count() or 1)
            del host
            b_prog = vs.Program(w["tree"](vs.Filter))
            nwords = sum((r + 63) // 64 for r in disk.rows)
            words = np.zeros(max(nwords, 1), dtype=np.uint64)
            counts = np.zeros(max(disk.nblocks, 1), dtype=np.uint32)
            bloom_first = {"workload": "C2: %s over %d rows, vocabulary rows in 1 block of 10 (hot_block_permille 100), on-disk blocks on pinned host memory" % (w["logsql"], b_rows)}
            keep = os.environ.get("VLSCAN_BLOOM_FIRST")
            for key, mode in (("one_go", "0"), ("bloom_first", "2")):
                os.environ["VLSCAN_BLOOM_FIRST"] = mode
                ctx.scan_batch(b_prog, disk, words, counts)
                sync_all()
                t0 = time.perf_counter()
                for _ in range(args.e2e_steps):
                    _, _, est = ctx.scan_batch(b_prog, disk, words, counts)
                sync_all()
                dt = (time.perf_counter() - t0) / args.e2e_steps
                bloom_first[key] = {"value": b_rows / dt, "unit": "rows/s", "ms_per_step": 1000 * dt, "h2d_bytes_per_step": int(est.h2d_bytes), "matched": int(counts.sum()),
                                    "staged_columns": int(est.staged_columns), "pruned_columns": int(est.pruned_columns)}
            if keep is None:
                os.environ.pop("VLSCAN_BLOOM_FIRST", None)
            else:
                os.environ["VLSCAN_BLOOM_FIRST"] = keep
            bloom_first["same_matches"] = bloom_first["one_go"]["matched"] == bloom_first["bloom_first"]["matched"]
            del disk
        except Exception as e:
            bloom_first = {"error": str(e)[:200]}

    if rank == 0:
        ms, steps = m["ms"], m["steps"]
        tr = ncu_traffic(args.workload, rows)
        out = {
            "metric": METRIC, "value": rows * world * steps / (ms / 1e3), "unit": "rows/s", "n_gpus": world, "steps": steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic (deterministic vlogsgenerator-shaped rows generated on the device, seed %d)" % SEED,
            "config": {"workload": "%s: %s over %d rows/GPU, %d fields" % (args.workload, wl["logsql"], rows, wl["fields"]), "rows_per_gpu": rows, "rows_per_block": wl["rows_per_block"],
                       "blocks_per_gpu": nb, "hot_block_permille": args.hot_block_permille, "hit_row_permille": args.hit_row_permille,
                       "l2": "inputs (%.1f GB/GPU) are far larger than the 126 MB L2; no flush between iterations" % (device_bytes / 1e9),
                       "parallelism": "blocks sharded over %d GPU(s); counters summed on the device every step, ONE NCCL all-reduce after the last step (inside the timed region)" % world if world > 1 else "1 GPU",
                       "gen_seconds": round(m["t_gen"], 2)},
            "rows_matched_per_gpu": int(st.rows_matched), "blocks_matched_per_gpu": int(st.blocks_matched),
            "algorithmic_bytes_per_step_per_gpu": int(m["step_bytes"]),
            "step_hbm_gbs_per_gpu": (m["step_bytes"] / 1e9) / (ms / steps / 1e3),
            "step_frac_of_peak": (m["step_bytes"] / 1e9) / (ms / steps / 1e3) / peak,
            "gpu_launches": int(st.gpu_launches) * steps,
            "clocks": m["clocks"],
            "roofline": {"bound": "hbm", "kernel": "k_substr_scan", "achieved": m["achieved"], "peak": peak, "unit": "GB/s", "frac": m["achieved"] / peak if peak else None,
                         "traffic": tr["dram_bytes_per_launch"] if tr else None,
                         "traffic_source": (tr.get("source") if tr else "no ncu --set full capture of this exact launch size under profiles/ (profiles/ncu_traffic_r02.json lists the ones that exist)"),
                         "peak_source": peak_src, "kernel_ms_per_launch": m["k_avg"], "algorithmic_bytes_per_launch": int(m["kbytes"]),
                         "kernel_share_of_step": m["share"]},
            "parity": parity, "e2e": e2e, "cpu_baseline": cpu, "cpu_baseline_post_zstd": cpu_post, "extra_workloads": extra or None, "e2e_bloom_first_staging": bloom_first,
        }
        if fallback_note:
            out["config"]["rows_note"] = "wanted %d rows/GPU: %s" % (want_rows, fallback_note)
        if numa:
            out["config"]["host_affinity"] = "each rank's threads bound to the NUMA node of its GPU (rank 0: node %d, %d CPUs)" % (numa["numa_node"], numa["cpus"])
        if m["totals"] is not None:
            out["allreduced_totals_over_timed_steps"] = {"rows": m["totals"][0], "rows_matched": m["totals"][1], "blocks_matched": m["totals"][2]}
        print(json.dumps(out), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
