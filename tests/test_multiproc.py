"""World-size-2 gloo test of the multi-GPU host logic (runs on CPU): read sharding by rank and stream, the
merge-step all-gather of packed contigs, and per-shard parity of what rank 0 receives.  The device work is done by
the TEST-ONLY emulation (tests/emu) here; on the B200 the same code path runs with NCCL (bench.py --gpus N)."""
import os
import sys

import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, emu_path, q, test_id):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import torch.distributed as dist
    from trust4_b200 import api, synth, dist as tdist
    import refharness as rh
    rh.use_tape("%s-rank%d" % (test_id, rank))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lib = api.Lib(emu_path, "t4emu_")
    lib.check(lib.init(0, 1 << 30))
    S = 3
    cl = synth.make_clones(20, 5)                               # shared repertoire
    rd = synth.sample_pairs(cl, 300, 150, 5000 + rank)          # rank-specific reads
    w = synth.build_workload(cl, rd)
    off, descs = synth.shard_workload(w, S)
    cfg = synth.run_cfg()
    sets = api.SeqSet.create_many(S, 9, lib)
    api.streams_run(sets, cfg, descs, off, w.pool, w.names, lib)
    buf, n = tdist.pack_contigs(lib, sets)
    gathered = tdist.allgather_contigs(buf)
    assert len(gathered) == world
    # every rank checks its own slice against the reference; rank 0 additionally checks what it received
    mine = tdist.format_output(tdist.unpack_contigs(gathered[rank]))
    for j in range(S):
        r = rh.RefSeqSet(9)
        r.run_descs(cfg, descs[int(off[j]):int(off[j + 1])].copy(), w.pool, w.names)
        assert r.output() == mine.get(j, b""), (rank, j)
    tot = sum(len(tdist.unpack_contigs(g)) for g in gathered)
    cnt = np.array([n], dtype=np.int64)
    import torch
    t = torch.from_numpy(cnt)
    dist.all_reduce(t)
    assert int(t.item()) == tot
    rh.end_tape()
    q.put((rank, tot))
    dist.destroy_process_group()


def test_two_rank_shard_and_allgather(emu_lib, ref, request):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 1000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, emu_lib.path, q, request.node.nodeid)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    res = sorted(q.get() for _ in range(2))
    assert res[0][1] == res[1][1] and res[0][1] > 0


def test_merge_oracle_on_packed_contigs(emu_lib, ref):
    """SURVEY.md 8e(2): the merged multi-GPU output is DEFINED as the reference's in-tree merge idiom
    (InputSeqSet + ChangeKmerLength(31) + RemoveRedundantSeq, main.cpp:2288-2294) over the concatenation of the shard
    contig sets in rank order.  What every rank holds after the all-gather (packed contigs) is enough to run that
    oracle: rebuilding the shard sets from the packed buffers gives the same merged set as merging the reference's
    own shard SeqSets.  (The merge itself stays reference CPU code in round 1 -- a 'next' row.)"""
    from trust4_b200 import api, synth, dist as tdist
    emu_lib.check(emu_lib.reset())
    cl = synth.make_clones(15, 8)
    rd = synth.sample_pairs(cl, 500, 150, 8)
    w = synth.build_workload(cl, rd)
    S = 4
    off, descs = synth.shard_workload(w, S)
    cfg = synth.run_cfg()
    sets = api.SeqSet.create_many(S, 9, emu_lib)
    api.streams_run(sets, cfg, descs, off, w.pool, w.names, emu_lib)
    buf, n = tdist.pack_contigs(emu_lib, sets)
    contigs = tdist.unpack_contigs(buf)
    assert len(contigs) == n
    rebuilt = [ref.set_from_contigs([c for c in contigs if c["set"] == j]) for j in range(S)]
    direct = []
    for j in range(S):
        r = ref.RefSeqSet(9)
        r.run_descs(cfg, descs[int(off[j]):int(off[j + 1])].copy(), w.pool, w.names)
        direct.append(r)
    m1, removed1 = ref.merge_sets(rebuilt)
    m2, removed2 = ref.merge_sets(direct)
    assert m1.output() == m2.output() and removed1 == removed2
    assert m1.size() == sum(1 for _ in contigs) - removed1 and removed1 >= 0


def test_pack_narrow_and_wide_counts(emu_lib):
    """Packed contig records: posWeight as u16 when every count fits, int32 otherwise (a contig with 70 000 copies of one read)."""
    sys.path.insert(0, ROOT)
    import numpy as np
    from trust4_b200 import api, dist as tdist
    emu_lib.check(emu_lib.reset())
    rng = np.random.default_rng(9)
    a = "".join("ACGT"[c] for c in rng.integers(0, 4, size=120))
    b = "".join("ACGT"[c] for c in rng.integers(0, 4, size=140))
    s = api.SeqSet(9, emu_lib)
    s.input_novel_read("IGHV1-2*01", a, 1, -1)
    s.input_novel_read("TRBV7-9*01", b, 1, -1)
    assert s.add_read(a, "IGHV", 0, -1, 5, 0, 0.9)[0] == 0
    for _ in range(70000):
        assert s.repeat_add_read(a) == 0
    buf, n = tdist.pack_contigs(emu_lib, [s])
    assert n == 2
    recs = tdist.unpack_contigs(buf)
    raw = buf.numpy()
    assert int(raw[28:32].view(np.uint32)[0]) == 0                       # contig 0: wide (int32) columns
    rb0 = int(raw[24:28].view(np.uint32)[0])
    assert int(raw[rb0 + 28:rb0 + 32].view(np.uint32)[0]) == 1           # contig 1: u16 columns
    assert recs[0]["pos_weight"].max() == 70002 and recs[1]["pos_weight"].max() == 1
    assert tdist.format_output(recs)[0] == s.output()
