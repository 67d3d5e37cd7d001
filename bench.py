#!/usr/bin/env python3
"""bench.py -- reads/sec assembled (150 bp PE) through the stage-1 AddRead loop on N B200s.

Workload (BASELINE.json configs[1]): 1 M synthetic 150 bp pairs (2 M reads) per GPU against the IMGT gene
set, k = 9, read-sharded into S independent streams (SURVEY.md 8e: contiguous shards of the sorted read
list, one SeqSet each; parity is per shard).  A step = one pass of the whole loop over the whole workload:
fresh streams -> stream kernel -> packed contigs (-> all-gather when N > 1).

  value      inputs resident in HBM, CUDA-event time over K steps (max over ranks)
  e2e        the same through t4_streams_run with pinned HOST buffers: H2D of records + reads, D2H of the per-read
             results AND of the packed contigs (the product of stage 1) inside the timed region
  roofline   the stream kernel (the hot kernel of a step): algorithmic bytes (SURVEY.md 8d) from the device counters /
             its CUDA-event duration, against MEASURED_PEAKS.json hbm_gbs
  roofline_probe   the dedicated k-mer probe kernel (t4_probe_kernel: GetHitsFromRead of all reads over the final sets)
  cpu_baseline / --impl reference: the reference's own SeqSet (oracle/_ref/libt4ref.so, compiled from the
             reference sources) driven over a uniform sample of the same shards on the host cores.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

REQUIRED_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                 "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "roofline_probe", "cpu_baseline")


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=int(os.environ.get("T4_BENCH_PAIRS", 1000000)))
    ap.add_argument("--clones", type=int, default=0, help="clonotypes (default pairs/50)")
    ap.add_argument("--streams", type=int, default=int(os.environ.get("T4_BENCH_STREAMS", 4096)))
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--ref-seconds", type=float, default=60.0, help="upper bound on the wall time of one reference sample")
    ap.add_argument("--ref-shards", type=int, default=2048, help="shards of one reference sample (a fixed uniform subset: the same "
                    "work in every run, so the figure is reproducible; bounded by --ref-seconds)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-probe", action="store_true")
    ap.add_argument("--deal", action="store_true", help="deal runs of identical reads round-robin to the streams instead of contiguous shards")
    ap.add_argument("--balance", default=os.environ.get("T4_BENCH_BALANCE", "cost"), choices=["reads", "cost"],
                    help="contiguous shards of equal read count, or of equal predicted cost (abundance model, synth.read_cost)")
    ap.add_argument("--dump-streams", default="", help="write per-stream cycles + features (npz) for cost-model calibration")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (rank 0) as DIR/<name>.npy: per read the "
                         "return code, strand and rescue code; per contig of a fixed seeded sample the consensus, posWeight and header")
    ap.add_argument("--config", type=int, default=1, choices=[1, 3, 4],
                    help="BASELINE.json configs[] index: 1 = bulk 150 bp PE (the metric's config), 3 = 10x-style barcoded single-end "
                         "reads (whole barcodes per stream), 4 = --repseq bulk TCR-seq 100 bp SE amplicons")
    ap.add_argument("--barcodes", type=int, default=int(os.environ.get("T4_BENCH_BARCODES", 1000)), help="config 3: cells per GPU (configs[3] full size: 6250)")
    ap.add_argument("--reads-per-barcode", type=int, default=2000)
    ap.add_argument("--reads", type=int, default=int(os.environ.get("T4_BENCH_READS", 2000000)), help="config 4: reads per GPU (configs[4] full size: 6250000)")
    ap.add_argument("--shard-by", default=os.environ.get("T4_BENCH_SHARD_BY", "gene"), choices=["rank", "gene"],
                    help="config 1.  gene (default): reads grouped by the gene of their rough annotation first, groups cut / packed into "
                         "streams of equal predicted cost -- a clonotype's reads meet in one SeqSet whatever their abundance rank (97.6 %% "
                         "of the V(D)J cores in one contig at S = 4096, same reads/s); rank: contiguous blocks of the sorted read list "
                         "(SURVEY.md 8e; 56 %%)")
    ap.add_argument("--no-quality", action="store_true", help="skip the assembly-quality figure (clonotypes spanned by one contig)")
    ap.add_argument("--kmer-stats", type=int, default=int(os.environ.get("T4_BENCH_KCOUNT", 1)),
                    help="configs 1/4: also time the 21-mer counting + per-read count statistics of the pre-processing on the device "
                         "(SURVEY.md 8f-3; `preprocess_kmer_stats`, outside value / e2e) and compare with the generator's figures; 0 = skip")
    ap.add_argument("--assign-pass", type=int, default=int(os.environ.get("T4_BENCH_ASSIGN", 1)),
                    help="config 1: also time the AssignRead pass over the finished sets (SURVEY.md 8f-2, main.cpp:2047-2118) -- a "
                         "separate figure (`assign_pass`), outside `value` and `e2e`; 0 = skip")
    args = ap.parse_args(argv)
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs writes what a timed step computed: it needs --steps >= 1")
    return args


def setup_of(args):
    """Per-config constants: read length, driver-loop configuration (main.cpp:1541-1568) and SeqSet setters."""
    from trust4_b200 import synth
    if args.config == 3:      # --barcode: hitLenRequired 13, barcode-salted index, per-barcode purge (main.cpp:1549-1560, 1846-1859)
        return {"L": 150, "cfg": synth.run_cfg(has_barcode=1, release_barcodes=1), "hit_len": 13, "consider_barcode": 1,
                "metric": "reads/sec assembled (150bp SE, 10x barcodes)"}
    if args.config == 4:      # --repseq = --trimLevel 2 --skipMateExtension: repetitiveData, k-change threshold halved (main.cpp:1567)
        return {"L": 100, "cfg": synth.run_cfg(repetitive=1, change_k_threshold=2048, first_read_len=100), "hit_len": 31, "consider_barcode": 0,
                "metric": "reads/sec assembled (100bp SE, --repseq)"}
    return {"L": 150, "cfg": synth.run_cfg(), "hit_len": 31, "consider_barcode": 0, "metric": "reads/sec assembled (150bp PE)"}


def dist_env():
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    return rank, world, local


def make_workload(args, rank, device):
    from trust4_b200 import synth
    if args.config == 3:
        nclones = args.clones or max(20, 2 * args.barcodes)
        cl = synth.make_clones(nclones, args.seed)
        rd, bc = synth.sample_single_cell(cl, args.barcodes, args.reads_per_barcode, 150, args.seed * 1000 + rank)
        w = synth.build_workload(cl, rd, device=device, barcode=bc)
        off, descs = synth.shard_workload(w, args.streams, balance=args.balance, align="barcode")
        return w, off, descs
    if args.config == 4:
        nclones = args.clones or max(20, args.reads // 50)
        cl = synth.make_clones(nclones, args.seed, chains=("TRB",))
        rd = synth.sample_amplicon(cl, args.reads, 100, args.seed * 1000 + rank, alpha=1.0)
        w = synth.build_workload(cl, rd, device=device, repseq=True)
        by_gene = (os.environ.get("T4_BENCH_CFG4_SHARD_BY", "rank") == "gene")
        off, descs = synth.shard_workload(w, args.streams, deal=args.deal, balance=args.balance, group="gene" if by_gene else "")
        args.streams = len(off) - 1
        make_workload.truth = (cl, rd)
        return w, off, descs
    nclones = args.clones or max(20, args.pairs // 50)
    cl = synth.make_clones(nclones, args.seed)                    # one repertoire for all ranks
    rd = synth.sample_pairs(cl, args.pairs, 150, args.seed * 1000 + rank)   # each rank sequences its own reads
    w = synth.build_workload(cl, rd, device=device)
    off, descs = synth.shard_workload(w, args.streams, deal=args.deal, balance=args.balance, group="gene" if args.shard_by == "gene" else "")
    args.streams = len(off) - 1
    make_workload.truth = (cl, rd)          # kept for the assembly-quality figure (bench/quality.py)
    return w, off, descs


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(max(mx))
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


def sample_order(n_shards):
    """Visit order of the reference sample: a fixed pseudo-random permutation, so that whatever prefix the time budget
    allows is a uniform sample over the shard index range (the sorted read list runs from cheap high-abundance shards
    to expensive singleton shards; a prefix of the index order would be biased)."""
    return np.random.default_rng(12345).permutation(n_shards)


def reference_sample(args, w, off, descs, budget_s, cores, keep=64):
    """The reference's SeqSet over a uniform sample of the shards on `cores` host threads for ~budget_s.
    reads/s = sum(reads of the sampled shards) / wall: with a uniform shard sample this estimates
    total_reads / total_cpu_time_on_cores for the whole workload."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import refharness as rh
    from trust4_b200 import synth
    if not rh.available():
        return None
    su = setup_of(args)
    cfg = su["cfg"]
    n_shards = len(off) - 1
    order = sample_order(n_shards)
    n_sample = min(n_shards, max(1, args.ref_shards))       # a fixed subset, not "whatever fits the budget"
    lock = threading.Lock()
    state = {"next": 0, "reads": 0, "shards": 0, "kept": {}, "assign_s": 0.0, "assign_reads": 0}
    t0 = time.perf_counter()

    def worker():
        while True:
            with lock:
                x = state["next"]
                if x >= n_sample or time.perf_counter() - t0 > budget_s:
                    return
                state["next"] += 1
            j = int(order[x])
            lo, hi = int(off[j]), int(off[j + 1])
            r = rh.RefSeqSet(9)
            if su["hit_len"] != 31:
                r.set_hit_len_required(su["hit_len"])
            if su["consider_barcode"]:
                rh.lib().t4ref_set_consider_barcode_in_hash(r.h, 1)
            out = r.run_descs(cfg, descs[lo:hi].copy(), w.pool, w.names)     # ctypes releases the GIL
            rec = None
            if x < keep:                                                     # the first `keep` of the order: full parity record
                rec = (out[1], out[3], r.output(), r.index_checksum())
                if args.config == 1 and args.assign_pass:                    # ... and the reference's AssignRead pass over the shard
                    ta = time.perf_counter()
                    lst = rh.assembled_list(out[1], out[3])
                    ext, ra, rs = rh.assign_pass(r, 17, descs[lo:hi], w.pool, lst, out[2])
                    rec = rec + ((lst, ra, rs, ext.output()),)
                    ext.close()
                    with lock:
                        state["assign_s"] += time.perf_counter() - ta
                        state["assign_reads"] += len(lst)
            r.close()
            with lock:
                state["reads"] += hi - lo
                state["shards"] += 1
                if rec is not None:
                    state["kept"][j] = rec

    th = [threading.Thread(target=worker) for _ in range(cores)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    el = time.perf_counter() - t0 - state["assign_s"] / max(1, cores)     # the AssignRead checks of the kept shards are not part of the loop's time
    reference_sample.kept = state["kept"]
    reference_sample.assign = {"reads": state["assign_reads"], "thread_seconds": state["assign_s"]}
    return {"value": state["reads"] / el, "unit": "reads/s", "cores": cores, "kind": "reference",
            "sample": "%d of %d read shards (%d reads), uniformly sampled over the shard index range (fixed permutation), %.1f s wall "
                      "on %d threads; oracle/_ref/libt4ref.so = reference SeqSet::AddRead/RepeatAddRead/InputNovelRead driven by the "
                      "restated main.cpp loop" % (state["shards"], n_shards, state["reads"], el, cores)}


DUMP_BYTES = 64 << 20


def dump_outputs(d, ret, strands, resc, packed, seed=0):
    """The results a caller of the timed step receives, as float arrays: t4_workload_results per read (return code, strand,
    rescue code; every read while they fit half of DUMP_BYTES, else a fixed seeded sample of reads, indices in read_index)
    and the packed contigs of every stream (t4_streams_pack_contigs), all of them or a fixed seeded sample within the rest of
    the budget.  Contig arrays: contig_header[c] = (index in pack order, set, slot, barcode, num_read, length),
    contig_consensus = the ASCII codes of the concatenated consensus strings, contig_pos_weight[sum(length), 4]."""
    os.makedirs(d, exist_ok=True)
    rng = np.random.default_rng(seed)
    n = len(ret)
    idx = np.arange(n)
    if n * 20 > DUMP_BYTES // 2:
        idx = np.sort(rng.choice(n, size=DUMP_BYTES // 2 // 28, replace=False))
        np.save(os.path.join(d, "read_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(d, "read_ret.npy"), ret[idx].astype(np.float64))
    np.save(os.path.join(d, "read_strand.npy"), strands[idx].astype(np.float32))
    np.save(os.path.join(d, "read_rescue.npy"), resc[idx].astype(np.float64))
    starts = []
    o = 0
    while o < len(packed):
        starts.append(o)
        o += int(packed[o + 24:o + 28].view(np.uint32)[0])
    budget = DUMP_BYTES - idx.nbytes * 3
    pick = np.arange(len(starts))
    if len(packed) * 3 > budget:        # one consensus byte -> 4 + 16 bytes of float32 output
        pick = np.sort(rng.choice(len(starts), size=max(1, int(len(starts) * budget / (3 * len(packed)))), replace=False))
    from trust4_b200 import dist as tdist
    hdr, cons, pw = [], [], []
    for c in pick:
        o = starts[c]
        rec = tdist.unpack_contigs(packed[o:o + int(packed[o + 24:o + 28].view(np.uint32)[0])])[0]
        hdr.append((c, rec["set"], rec["slot"], rec["barcode"], rec["num_read"], len(rec["consensus"])))
        cons.append(np.frombuffer(rec["consensus"].encode(), dtype=np.uint8))
        pw.append(rec["pos_weight"])
    np.save(os.path.join(d, "contig_header.npy"), np.array(hdr, dtype=np.float64).reshape(-1, 6))
    np.save(os.path.join(d, "contig_consensus.npy"), np.concatenate(cons or [np.zeros(0, np.uint8)]).astype(np.float32))
    np.save(os.path.join(d, "contig_pos_weight.npy"), np.concatenate(pw or [np.zeros((0, 4), np.int32)]).astype(np.float32))


def build_line(args, config, value, ms_per_step, clocks, e2e, launches, roofline, roofline_probe, cpu, extra, metric="reads/sec assembled (150bp PE)"):
    """The ONE JSON line of the contract.  Kept as a pure function so that a unit test can assert its keys."""
    line = {"metric": metric, "value": value, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "roofline_probe": roofline_probe, "cpu_baseline": cpu}
    line.update(extra)
    for k in REQUIRED_KEYS:
        assert k in line, k
    return line


def main():
    args = parse()
    rank, world, local = dist_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    cores = os.cpu_count() or 1
    mode = "grouped by annotated gene, groups packed by predicted cost" if args.shard_by == "gene" else "dealt round-robin" if args.deal else ("in contiguous blocks of the sorted list, block sizes equalising the predicted cost (abundance model)"
                                                   if args.balance == "cost" else "in contiguous blocks of the sorted list, equal read counts")
    if args.config == 3:
        args.streams = min(args.streams, args.barcodes)
        wtxt = ("configs[3] shape: %d cell barcodes x %d synthetic 150bp SE reads per GPU (configs[3] full size is 6250 barcodes per GPU), "
                "hitLenRequired 13, barcode-salted index, whole barcodes per stream (%d streams per GPU, SURVEY.md 8e), finished barcodes purged"
                % (args.barcodes, args.reads_per_barcode, args.streams))
    elif args.config == 4:
        wtxt = ("configs[4] shape: %d synthetic 100bp SE TRB amplicon reads per GPU (--repseq: repetitiveData, V-gene pseudo barcodes; configs[4] "
                "full size is 6.25 M per GPU), read-sharded into %d streams per GPU (%s)" % (args.reads, args.streams, mode))
    else:
        wtxt = ("configs[1]: %d synthetic 150bp PE pairs (%d reads) per GPU vs human_IMGT+C gene pool, k=9, "
                "read-sharded into %d streams per GPU (runs of identical reads %s; one SeqSet each, per-shard parity, SURVEY.md 8e)"
                % (args.pairs, 2 * args.pairs, args.streams, mode))
    su = setup_of(args)
    L = su["L"]
    config = {"workload": wtxt, "baseline_config": args.config,
              "pairs_per_gpu": args.pairs if args.config == 1 else None, "streams_per_gpu": args.streams, "kmer": 9, "read_len": L, "shard_balance": "deal" if args.deal else args.balance,
              "l2": "inputs (>= 400 MB of reads + records, GBs of stream state) exceed the 126 MB L2",
              "sharding": "rank r sequences its own reads of the shared repertoire; no data-path collective; "
                          "N>1: one NCCL all-gather of the packed per-rank contig sets per step (merge step)"}

    if args.impl == "reference":
        if rank != 0:
            return
        gen_dev = None
        try:
            import torch
            if torch.cuda.is_available():
                gen_dev = torch.device("cuda", local)      # workload preparation only (21-mer statistics); the arm itself is CPU
        except Exception:
            gen_dev = None
        w, off, descs = make_workload(args, 0, gen_dev)
        per_step = args.ref_seconds
        vals = []
        for it in range(args.warmup + args.steps):
            s = reference_sample(args, w, off, descs, per_step, cores, keep=0)
            if s is None:
                print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libt4ref.so not built"}))
                return
            if it >= args.warmup:
                vals.append(s)
        v = float(np.mean([x["value"] for x in vals]))
        n_reads = len(descs)
        line = {"impl": "reference", "metric": su["metric"], "value": v, "unit": "reads/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n_reads / v, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": config,
                "cpu_baseline": dict(vals[-1], value=v),
                "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    from trust4_b200 import api, synth
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = api.default_lib()
    lib.check(lib.init(local, 0))
    dev = torch.device("cuda", local)

    t_gen = time.perf_counter()
    w, off, descs = make_workload(args, rank, dev)
    t_gen = time.perf_counter() - t_gen
    torch.cuda.empty_cache()
    n_reads = len(descs)
    S = args.streams
    cfg = su["cfg"]
    names_arr = api._names_array(w.names)
    off64 = np.ascontiguousarray(off, dtype=np.int64)

    # pinned host copies for the e2e leg
    pin_descs = torch.from_numpy(descs.view(np.uint8).reshape(-1).copy()).pin_memory()
    pin_pool = torch.from_numpy(w.pool.copy()).pin_memory()
    ret = torch.zeros(n_reads, dtype=torch.int32).pin_memory()
    strands = torch.zeros(n_reads, dtype=torch.int8).pin_memory()
    resc = torch.zeros(n_reads, dtype=torch.int32).pin_memory()
    h2d_bytes = pin_descs.numel() + pin_pool.numel() + S * 256

    wl = lib.workload_upload(pin_descs.data_ptr(), n_reads, pin_pool.data_ptr(), pin_pool.numel(), names_arr, len(w.names))
    if not wl:
        raise RuntimeError(lib.err())
    handles = (C.c_void_p * S)()

    merged = {"bytes": 0, "contigs": 0, "pack_bytes": 0}
    pack = {"buf": None, "host": None}

    def pack_contigs():
        """Stage-1 product: every live contig of this rank, packed on the device into one buffer."""
        need, nc = C.c_size_t(), C.c_int64()
        lib.check(lib.streams_pack_contigs(handles, S, None, 0, C.byref(need), C.byref(nc)))
        if pack["buf"] is None or pack["buf"].numel() < need.value:
            pack["buf"] = torch.empty(int(need.value * 1.1) + 1024, dtype=torch.uint8, device=dev)
        lib.check(lib.streams_pack_contigs(handles, S, pack["buf"].data_ptr(), pack["buf"].numel(), C.byref(need), C.byref(nc)))
        merged["contigs"] = int(nc.value)
        merged["pack_bytes"] = int(need.value)
        return pack["buf"][: need.value]

    def merge_exchange(buf):
        """Merge step of a read-sharded multi-GPU run: all-gather the packed contig sets over NCCL."""
        if world == 1:
            return
        from trust4_b200 import dist as tdist
        parts = tdist.allgather_contigs(buf)
        merged["bytes"] = int(sum(p.numel() for p in parts))

    def step_resident():
        lib.check(lib.reset())
        lib.check(lib.seqsets_create_ex(S, 9, su["hit_len"], su["consider_barcode"], handles))
        lib.check(lib.streams_run_resident(handles, S, cfg.ctypes.data, wl, off64.ctypes.data, None))
        merge_exchange(pack_contigs())

    def step_e2e():
        lib.check(lib.reset())
        lib.check(lib.seqsets_create_ex(S, 9, su["hit_len"], su["consider_barcode"], handles))
        lib.check(lib.streams_run(handles, S, cfg.ctypes.data, pin_descs.data_ptr(), off64.ctypes.data, pin_pool.data_ptr(),
                                  pin_pool.numel(), names_arr, len(w.names), ret.data_ptr(), strands.data_ptr(), resc.data_ptr()))
        buf = pack_contigs()
        if pack["host"] is None or pack["host"].numel() < buf.numel():
            pack["host"] = torch.empty(int(buf.numel() * 1.1) + 1024, dtype=torch.uint8).pin_memory()
        pack["host"][: buf.numel()].copy_(buf, non_blocking=True)          # the contigs cross PCIe inside the timed region
        merge_exchange(buf)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()
    if args.warmup > 0 and lib.streams_error(handles, S):
        raise RuntimeError("device error after warm-up: " + lib.err())
    sampler = ClockSampler(local) if rank == 0 else None
    ms = timed(step_resident, args.steps)
    clocks = sampler.stop() if sampler else None
    lib.check(lib.workload_results(wl, ret.data_ptr(), strands.data_ptr(), resc.data_ptr()))
    assembled = int((ret >= 0).sum().item() + (resc >= 0).sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ret.numpy(), strands.numpy(), resc.numpy(), pack["buf"][: merged["pack_bytes"]].cpu().numpy())

    # kernel-only duration of the stream kernel (one launch per step) for the roofline
    lib.check(lib.reset())
    lib.check(lib.seqsets_create_ex(S, 9, su["hit_len"], su["consider_barcode"], handles))
    torch.cuda.synchronize()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0 = np.zeros(api.N_COUNTERS, dtype=np.uint64)
    lib.check(lib.last_counters(c0.ctypes.data))
    k0.record()
    lib.check(lib.streams_run_resident(handles, S, cfg.ctypes.data, wl, off64.ctypes.data, None))
    k1.record()
    torch.cuda.synchronize()
    kernel_ms = k0.elapsed_time(k1)
    c1 = np.zeros(api.N_COUNTERS, dtype=np.uint64)
    lib.check(lib.last_counters(c1.ctypes.data))
    dc = (c1 - c0).astype(np.float64)
    cyc = np.zeros(S, dtype=np.uint64)
    lib.check(lib.streams_cycles(handles, S, cyc.ctypes.data))
    cycf = cyc.astype(np.float64)
    if args.dump_streams and rank == 0:
        lib.check(lib.workload_results(wl, ret.data_ptr(), strands.data_ptr(), resc.data_ptr()))
        np.savez_compressed(args.dump_streams, cycles=cyc, off=off64, flags=descs["flags"], min_cnt=descs["min_cnt"], med=w.med_cnt,
                            ret=ret.numpy().copy())
    balance = {"mean_ms": float(cycf.mean() / 1.965e6), "max_ms": float(cycf.max() / 1.965e6), "p50_ms": float(np.median(cycf) / 1.965e6),
               "p99_ms": float(np.percentile(cycf, 99) / 1.965e6), "reads_per_stream_min_max": [int(np.diff(off64).min()), int(np.diff(off64).max())],
               "by_decile_of_stream_index_ms": [float(x.mean() / 1.965e6) for x in np.array_split(cycf, 10)]}
    # SURVEY.md 8d: probe ceil(L/4) + sum(8 + 8 c_j) + 16 sum c_j'; chain 2 x 16 sum c_j'; commit 8 L per assembled read
    b_probe = dc[5] + 8 * dc[2] + 8 * dc[3] + 16 * dc[4]
    b_chain = 32 * dc[4]
    b_commit = 8.0 * L * assembled
    alg_bytes = b_probe + b_chain + b_commit
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

    def ncu_traffic(fname):
        """DRAM bytes (read + write) of a kernel from a committed ncu --set full raw page of the default workload."""
        try:
            if args.config != 1 or args.pairs != 1000000 or args.streams != 4096 or args.deal:
                return None
            import csv
            rows = list(csv.reader(open(os.path.join(ROOT, "profiles", fname))))
            hdr, units, vals = rows[0], rows[1], rows[2]
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
            return sum(float(vals[hdr.index(m)]) * scale[units[hdr.index(m)]] for m in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
        except Exception:
            return None

    traffic_file = "r2_stream_kernel_full_raw.csv" if os.path.exists(os.path.join(ROOT, "profiles", "r2_stream_kernel_full_raw.csv")) else "r1_stream_kernel_full_raw.csv"
    traffic = ncu_traffic(traffic_file)
    ach = alg_bytes / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "t4_stream_kernel", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "traffic_source": ("profiles/%s (ncu --set full, same workload)" % traffic_file) if traffic else None,
                "algorithmic_bytes_total": alg_bytes, "peak_source": peak_src, "kernel_ms": kernel_ms,
                "algorithmic_bytes": {"probe": b_probe, "chain": b_chain, "commit": b_commit},
                "per_read": {"lookups": dc[2] / n_reads, "hits": dc[4] / n_reads, "overlaps_scored": dc[6] / n_reads, "gap_dps": dc[7] / n_reads,
                             "extend_dps": dc[1] / n_reads, "overlaps_extended": dc[16] / n_reads},
                "extend_split": dict(zip(["overhang_bits", "settle", "deferred_dps"], [round(float(x), 4) for x in (dc[17:20] / max(1.0, dc[17:20].sum()))])),
                "stream_balance": balance, "phase_share": dict(zip(["other", "probe", "hit_sort", "chains", "score", "extend", "decide_commit", "novel_repeat_consensus"],
                                        [round(float(x), 4) for x in (dc[8:16] / max(1.0, dc[8:16].sum()))]))}

    # ---- the dedicated probe kernel over the final sets of this very run
    roofline_probe = None
    if not args.no_probe:
        cap = int(2.2e9 if n_reads >= 1000000 else max(1 << 22, 2000 * n_reads))
        st = np.zeros(8, dtype=np.uint64)
        hits = None
        for attempt in range(2):
            hits = lib.hits_create(n_reads, cap)
            if not hits:
                raise RuntimeError(lib.err())
            lib.check(lib.streams_get_hits(handles, S, wl, off64.ctypes.data, 0, None, hits))      # warm-up + sizing
            r = lib.hits_stats(hits, st.ctypes.data)
            if r == api.T4_E_NOMEM and attempt == 0:
                need = int(lib.err().split(":")[1].split()[0])
                lib.hits_free(hits)
                cap = int(need * 1.02) + 1024
                continue
            lib.check(r)
            break
        pms = []
        for _ in range(3):
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            p0.record()
            lib.check(lib.streams_get_hits(handles, S, wl, off64.ctypes.data, 0, None, hits))
            p1.record()
            torch.cuda.synchronize()
            pms.append(p0.elapsed_time(p1))
        lib.check(lib.hits_stats(hits, st.ctypes.data))
        lib.hits_free(hits)
        pm = float(np.median(pms))
        a = float(st[4]) / (pm * 1e-3) / 1e9
        a16 = float(st[5]) / (pm * 1e-3) / 1e9
        roofline_probe = {"bound": "hbm", "kernel": "t4_probe_kernel (+ t4_bucket_kernel): GetHitsFromRead of every read over the final contig sets, warp per read",
                          "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak, "kernel_ms": pm, "kernel_ms_all": pms,
                          "algorithmic_bytes": int(st[4]),
                          "algorithmic_bytes_note": "SURVEY.md 8d with the 8-byte hit key this kernel writes: ceil(L/4) + 8 lookups + 8 postings + 8 hits",
                          "achieved_with_16B_hits": a16, "frac_with_16B_hits": a16 / peak,
                          "hits": int(st[0]), "lookups": int(st[1]), "postings": int(st[2]), "reads_per_s": n_reads / (pm * 1e-3),
                          "traffic": ncu_traffic("r2_probe_kernel_full_raw.csv"),
                          "l2_note": "reads are visited set by set, so directory and postings sectors of a set are re-used from L2"}

    # ---- e2e leg, with separately timed copies
    step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    e2e_assembled = int((ret >= 0).sum().item() + (resc >= 0).sum().item())
    assert e2e_assembled == assembled, (e2e_assembled, assembled)
    d2h_bytes = n_reads * 9 + merged["pack_bytes"]
    dpool = torch.empty(pin_pool.numel() + pin_descs.numel(), dtype=torch.uint8, device=dev)
    x0, x1, x2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    torch.cuda.synchronize()
    x0.record()
    dpool[: pin_pool.numel()].copy_(pin_pool, non_blocking=True)
    dpool[pin_pool.numel():].copy_(pin_descs, non_blocking=True)
    x1.record()
    pack["host"][: merged["pack_bytes"]].copy_(pack["buf"][: merged["pack_bytes"]], non_blocking=True)
    x2.record()
    torch.cuda.synchronize()
    copies = {"h2d_ms": x0.elapsed_time(x1), "h2d_gbs": (pin_pool.numel() + pin_descs.numel()) / x0.elapsed_time(x1) / 1e6,
              "d2h_contigs_ms": x1.elapsed_time(x2), "d2h_contigs_gbs": merged["pack_bytes"] / max(1e-6, x1.elapsed_time(x2)) / 1e6}
    del dpool


    # ---- the AssignRead pass over the finished sets (SURVEY.md 8f-2; main.cpp:2047-2118): its own figure, outside value / e2e
    assign_fig, assign_obj = None, None
    if args.config == 1 and args.assign_pass:
        try:
            ams = []
            st4 = np.zeros(4, dtype=np.uint64)
            for _ in range(2):                   # the second run is the timed one (the first also warms the allocator)
                if assign_obj:
                    lib.assign_free(assign_obj)
                torch.cuda.synchronize()
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                assign_obj = lib.streams_assign_reads(handles, S, wl, off64.ctypes.data, 17, 0, None)
                if not assign_obj:
                    raise RuntimeError(lib.err())
                a1.record()
                torch.cuda.synchronize()
                ams.append(a0.elapsed_time(a1))
            lib.check(lib.assign_stats(assign_obj, st4.ctypes.data))
            assign_fig = {"what": "extendedSeq(17).InputSeqSet per stream + AssignRead of every assembled read (worker CTAs over the whole "
                                  "GPU) + RecomputePosWeight; three launches of t4_aux_kernel",
                          "ms": ams[-1], "ms_all": ams, "reads": int(st4[0]), "assign_calls": int(st4[1]), "assigned": int(st4[2]),
                          "worker_ctas": int(st4[3]), "reads_per_s": float(st4[0]) / (ams[-1] * 1e-3), "kmer": 17}
        except Exception as ex:      # a separate figure: never let it break the headline measurement
            assign_fig = {"error": str(ex)[:300]}


    # ---- 21-mer counting + per-read count statistics of the pre-processing (SURVEY.md 8f-3), its own figure
    kc_fig = None
    if args.config in (1, 4) and args.kmer_stats and rank == 0:
        try:
            dpool2 = torch.from_numpy(w.pool).to(dev)
            doff = torch.from_numpy(w.descs["seq_off"].astype(np.int64)).to(dev)
            dlen = torch.from_numpy(w.descs["len"].astype(np.int32)).to(dev)
            inst = int(np.maximum(w.descs["len"].astype(np.int64) - 20, 0).sum())
            tb = int(lib.kmer_count_table_bytes(max(1 << 20, inst // 2)))       # capacity hint: half the instances (distinct k-mers are far fewer)
            table = torch.empty(tb, dtype=torch.uint8, device=dev)
            omn = torch.empty(n_reads, dtype=torch.int32, device=dev)
            omed = torch.empty(n_reads, dtype=torch.int32, device=dev)
            oavg = torch.empty(n_reads, dtype=torch.float32, device=dev)
            kms = []
            for _ in range(3):
                q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                q0.record()
                lib.check(lib.kmer_count_stats_device(dpool2.data_ptr(), None, doff.data_ptr(), dlen.data_ptr(), n_reads, 21, table.data_ptr(), tb,
                                                      omn.data_ptr(), omed.data_ptr(), oavg.data_ptr(), None, None))
                q1.record()
                torch.cuda.synchronize()
                kms.append(q0.elapsed_time(q1))
            ks = np.zeros(4, dtype=np.uint64)
            lib.check(lib.kmer_count_table_stats(table.data_ptr(), tb, ks.ctypes.data))
            km = float(np.median(kms))
            eq_min = bool((omn.cpu().numpy() == w.descs["min_cnt"]).all())
            eq_med = bool((omed.cpu().numpy() == w.med_cnt).all()) if w.med_cnt is not None else None
            kc_fig = {"what": "KmerCount(21): AddCount of every read + GetCountStatsAndTrim (no trimming) -> minCnt / medianCnt / avgCnt per read; "
                              "two launches of t4_kcount_kernel over one HBM hash table",
                      "ms": km, "ms_all": kms, "reads_per_s": n_reads / (km * 1e-3), "kmers": int(ks[0]), "distinct_kmers": int(ks[1]),
                      "table_slots": int(ks[2]), "table_overflow": bool(ks[3]), "kmers_per_s": float(ks[0]) / (km * 1e-3),
                      "equals_generator_min_cnt": eq_min, "equals_generator_median_cnt": eq_med,
                      "note": "the workload generator's own statistics come from torch.unique/sort (library calls); parity against the "
                              "reference's KmerCount is tests/test_gpu_parity.py::test_gpu_kmer_count_stats"}
            del dpool2, table
        except Exception as ex:
            kc_fig = {"error": str(ex)[:300]}

    value = world * n_reads * args.steps / (ms * 1e-3)
    e2e = world * n_reads * args.steps / (ms_e2e * 1e-3)
    quality_fig = None
    if rank == 0 and not args.no_quality and args.config in (1, 4) and getattr(make_workload, "truth", None) is not None:
        # what the sharding costs in contiguity: clonotypes whose V(D)J core lies inside ONE contig of this rank's output
        try:
            sys.path.insert(0, os.path.join(ROOT, "bench"))
            import quality
            torch.cuda.synchronize()
            tq = time.perf_counter()
            codes, coff, ncont = quality.contigs_from_packed(pack["host"][: merged["pack_bytes"]].numpy())
            cl_, rd_ = make_workload.truth
            if args.config == 4:    # amplicon reads all start at the C primer: the 200 bp window is never covered, so count
                quality_fig = quality.recovered_fraction(cl_, rd_, codes, coff)     # clonotypes whose junction 24-mer is in a contig
            else:
                quality_fig = quality.spanning_fraction(cl_, rd_, codes, coff)
            quality_fig.update(contigs=ncont, contig_bases=int(len(codes)), streams=S, seconds=time.perf_counter() - tq)
        except Exception as ex:
            quality_fig = {"error": str(ex)[:200]}
    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            cpu = reference_sample(args, w, off, descs, args.ref_seconds, cores)
        # the CPU baseline leg doubles as a full-scale parity check: for the first shards of the sample the reference's return
        # codes, rescue codes, Output text and index checksum must equal what the GPU produced in the e2e leg
        parity = None
        try:
            kept = getattr(reference_sample, "kept", {}) if cpu else {}
            if kept:
                gret, gres = ret.numpy(), resc.numpy()
                bad = []
                ga = gs = None
                abad, achecked = [], 0
                if assign_obj:
                    ga = np.zeros((n_reads, 8), dtype=np.int32)
                    gs = np.zeros(n_reads, dtype=np.float64)
                    lib.check(lib.assign_results(assign_obj, ga.ctypes.data, gs.ctypes.data))
                for j, rec in kept.items():
                    rret, rres, rout, rsum = rec[:4]
                    lo, hi = int(off[j]), int(off[j + 1])
                    g = api.SeqSet(9, lib, handles[j])
                    ok = (gret[lo:hi] == rret).all() and (gres[lo:hi] == rres).all() and g.output() == rout and g.index_checksum() == rsum
                    if not ok:
                        bad.append(int(j))
                    if ga is not None and len(rec) > 4:
                        lst, ra, rs, eout = rec[4]
                        gj = ga[lo:hi][lst]
                        okr = ra[:, 0] >= 0
                        ge = api.SeqSet(17, lib, lib.assign_extended_set(assign_obj, int(j)))
                        oka = ((gj[:, 0] == ra[:, 0]).all() and (gj[okr] == ra[okr]).all() and (gs[lo:hi][lst][okr] == rs[okr]).all()
                               and ge.output() == eout)
                        ge.h = None
                        achecked += 1
                        if not oka:
                            abad.append(int(j))
                parity = {"shards_checked": len(kept), "checked": "return codes, rescue codes, Output text, index checksum",
                          "equal_reference": len(bad) == 0, "bad_shards": bad[:8]}
                if assign_fig is not None and "error" not in assign_fig:
                    ra_ = getattr(reference_sample, "assign", None) or {}
                    assign_fig["parity_spot_check"] = {"shards_checked": achecked, "equal_reference": achecked > 0 and len(abad) == 0, "bad_shards": abad[:8],
                                                       "checked": "per read: contig, coordinates, strand, matchCnt, similarity; per stream: Output text of the extended set after RecomputePosWeight"}
                    if ra_.get("thread_seconds"):
                        assign_fig["cpu_reference"] = {"reads_per_s_per_thread": ra_["reads"] / ra_["thread_seconds"], "reads": ra_["reads"],
                                                       "note": "reference InputSeqSet + AssignRead + RecomputePosWeight over the same sampled shards, per host thread (the reference runs this pass on -t threads, main.cpp:2086-2116)"}
        except Exception as ex:      # never let the checker break the measurement
            parity = {"error": str(ex)[:200]}
        line = build_line(
            args, config, value, ms / args.steps, clocks,
            {"value": e2e, "unit": "reads/s", "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes),
             "ms_per_step": ms_e2e / args.steps, "copies": copies,
             "d2h_note": "per-read return codes (9 B/read) + the packed contigs of every stream (consensus, posWeight, names)"},
            # init + stream kernel + pack-size + pack per step
            4 * args.steps, roofline, roofline_probe, cpu,
            {"assembled_reads": assembled, "reads_per_gpu": n_reads, "contigs_per_gpu": merged["contigs"], "parity_spot_check": parity,
             "assembly_quality": quality_fig, "assign_pass": assign_fig, "preprocess_kmer_stats": kc_fig,
             "merge_allgather": merged if world > 1 else None, "workload_gen_s": t_gen,
             "threads_per_stream": int(os.environ.get("T4_NT", 128))}, metric=su["metric"])
        print(json.dumps(line))
    if assign_obj:
        lib.assign_free(assign_obj)
    lib.workload_free(wl)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
