"""Parity checks shared by the emulation (CPU, tests/emu) and GPU test modules.  `lib` is an api.Lib."""
import gzip
import os

import numpy as np

from trust4_b200 import api, synth
import refharness
import tracereplay as tr

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def gold_trace(name):
    return tr.load_trace(os.path.join(GOLD, name + ".trace.gz"))


def gold_raw(name):
    return gzip.open(os.path.join(GOLD, name + "_raw.out.gz")).read()


def check_trace_replay(lib, name):
    """Every SeqSet call of a real trust4 run, one C-ABI call each: return values, strand outputs and the
    final Output text must equal what the reference binary produced."""
    lib.check(lib.reset())
    s, bad = tr.replay(gold_trace(name), lambda k: api.SeqSet(k, lib))
    assert not bad, bad[:1]
    assert s.output() == gold_raw(name)


def small_workload(seed, nclones=25, npairs=400, L=150):
    cl = synth.make_clones(nclones, seed)
    rd = synth.sample_pairs(cl, npairs, L, seed)
    return synth.build_workload(cl, rd)


def check_batch_vs_ref(lib, ref, seed, n_shards, nclones=25, npairs=400, cfg=None, deal=False, group="", c_mode=None):
    """t4_streams_run over read shards == the reference SeqSet driven by the restated loop, per shard.
    c_mode: shard with the library's t4_shard_reads (what the batch drop-in calls) instead of synth.shard_workload."""
    lib.check(lib.reset())
    w = small_workload(seed, nclones, npairs)
    cfg = cfg if cfg is not None else synth.run_cfg()
    if c_mode is not None:
        off, descs, _ = api.shard_reads(w.descs, n_shards, c_mode, lib)
    else:
        off, descs = synth.shard_workload(w, n_shards, deal=deal, balance="cost" if group else "reads", group=group)
    n_shards = len(off) - 1
    k = 9
    sets = api.SeqSet.create_many(n_shards, k, lib)
    ret, strands, resc = api.streams_run(sets, cfg, descs, off, w.pool, w.names, lib)
    for j in range(n_shards):
        lo, hi = int(off[j]), int(off[j + 1])
        r = ref.RefSeqSet(k)
        _, rret, rstr, rresc = r.run_descs(cfg, descs[lo:hi].copy(), w.pool, w.names)
        assert (rret == ret[lo:hi]).all(), ("ret", j, np.flatnonzero(rret != ret[lo:hi])[:5])
        assert (rstr == strands[lo:hi]).all(), ("strand", j)
        assert (rresc == resc[lo:hi]).all(), ("rescue", j)
        assert r.output() == sets[j].output(), ("contigs", j)
        assert r.index_checksum() == sets[j].index_checksum(), ("index", j)
        assert r.size() == sets[j].size()
    return int((ret >= 0).sum())


_canon4 = refharness.canon4
canon_hits = refharness.canon_hits


def _ragged_records(rng, sources, n, kmer=9):
    """Probe records of mixed lengths (shorter than k .. 400 bp: the probe tiles 288 positions), N's, all strand modes."""
    reads, descs = [], np.zeros(n, dtype=synth.READ_DESC)
    off = 0
    for i in range(n):
        src = sources[int(rng.integers(len(sources)))]
        L = int(rng.choice([5, kmer - 1, kmer, kmer + 1, 31, 64, 100, 144, 145, 150, 152, 153, 200, 290, 400]))
        while len(src) < L:
            src = src + sources[int(rng.integers(len(sources)))]
        a = int(rng.integers(0, len(src) - L + 1))
        s = list(src[a:a + L])
        for _ in range(int(rng.integers(0, 4))):
            s[int(rng.integers(L))] = "ACGTN"[int(rng.integers(5))]
        if rng.random() < 0.15:
            p0 = int(rng.integers(L))
            s[p0:p0 + 14] = list("A" * len(s[p0:p0 + 14]))                             # homopolymer: equal consecutive k-mers
        s = "".join(s)
        assert len(s) == L
        if rng.random() < 0.4:
            s = "".join({"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}[c] for c in reversed(s))
        reads.append(s)
        descs[i]["seq_off"] = off
        descs[i]["len"] = L
        descs[i]["barcode"] = -1
        descs[i]["strand_in"] = int(rng.choice([0, 0, 1, -1]))
        off += L
    pool = np.frombuffer(("".join(reads) + "\0" * 16).encode(), dtype=np.uint8).copy()
    return reads, descs, pool


def check_probe_batch(lib, ref, seed=41, n_shards=5, sample=160):
    """t4_streams_get_hits (the grid-wide warp-per-read probe: 2-bit packed reads, directory + postings over frozen sets)
    against SeqSet::GetHitsFromRead of the reference on the same sets: hit multisets per record, for the assembled reads
    of every shard and for ragged records (lengths 5..400, N's, homopolymers, both strands, strand -1/0/+1 modes)."""
    lib.check(lib.reset())
    w = small_workload(seed, 25, 500)
    cfg = synth.run_cfg()
    off, descs = synth.shard_workload(w, n_shards)
    sets = api.SeqSet.create_many(n_shards, 9, lib)
    api.streams_run(sets, cfg, descs, off, w.pool, w.names, lib)
    refs = []
    for j in range(n_shards):
        r = ref.RefSeqSet(9)
        r.run_descs(cfg, descs[int(off[j]):int(off[j + 1])].copy(), w.pool, w.names)
        assert r.index_checksum() == sets[j].index_checksum()
        refs.append(r)
    rng = np.random.default_rng(seed)
    # (1) the workload's own records
    wl = api.Workload(descs, w.pool, w.names, lib)
    hits = api.Hits(len(descs), 4 << 20, lib)
    api.streams_get_hits(sets, wl, off, hits)
    st = hits.stats()
    assert st["records"] == len(descs) and st["hits"] > 1000 and st["unsupported"] == 0
    reads = w.pool[: len(w.descs) * w.L].reshape(-1, w.L)
    total = 0
    for i in rng.choice(len(descs), size=min(sample, len(descs)), replace=False):
        j = int(np.searchsorted(off, i, side="right") - 1)
        d = descs[i]
        rd = bytes(w.pool[int(d["seq_off"]):int(d["seq_off"]) + int(d["len"])]).decode()
        hr = _canon4(refs[j].get_hits(rd, int(d["strand_in"]), int(d["barcode"])))
        hg, _ = hits.fetch(int(i))
        hg = _canon4(hg)
        assert hr.shape == hg.shape and (hr == hg).all(), ("probe", int(i), j, hr.shape, hg.shape)
        total += len(hr)
    assert total > 100
    wl.close()
    # (2) ragged records against the same frozen sets
    srcs = []
    for j in range(n_shards):
        for line in sets[j].output().split(b"\n"):
            if line and line[:1] in b"ACGT" and len(line) > 60 and b" " not in line:
                srcs.append(line.decode())
    assert len(srcs) >= n_shards
    n = 300
    rreads, rdescs, rpool = _ragged_records(rng, srcs, n)
    roff = np.linspace(0, n, n_shards + 1).astype(np.int64)
    wl = api.Workload(rdescs, rpool, [], lib)
    for skip in (0, 1):
        api.streams_get_hits(sets, wl, roff, hits, allow_total_skip=skip)
        st = hits.stats()
        assert st["records"] == n
        nz = 0
        for i in range(n):
            j = int(np.searchsorted(roff, i, side="right") - 1)
            hr = _canon4(refs[j].get_hits(rreads[i], int(rdescs[i]["strand_in"]), -1, bool(skip)))
            hg, _ = hits.fetch(i)
            hg = _canon4(hg)
            assert hr.shape == hg.shape and (hr == hg).all(), ("ragged", i, len(rreads[i]), int(rdescs[i]["strand_in"]), hr.shape, hg.shape)
            nz += len(hr) > 0
        assert nz > n // 3
    wl.close()
    hits.close()


def check_stage_parity(lib, ref, name="synth2k", every=97, max_checks=60):
    """k-mer hits (after SortHits) and scored overlaps of individual reads against a frozen snapshot:
    replay the golden trace on both sides and compare the stage outputs at sampled AddRead calls."""
    lib.check(lib.reset())
    ops = gold_trace(name)
    g = None
    r = None
    checks = 0
    for i, t in enumerate(ops):
        if t[0] == "A" and i % every == 0 and checks < max_checks:
            read, sin = t[1], int(t[3])
            hr = canon_hits(r.get_hits(read, sin))
            hg = g.get_hits(read, sin)
            assert hr.shape == hg.shape and (hr == hg).all(), ("hits", i)
            n1, o1, s1 = r.get_overlaps(read, sin)
            n2, o2, s2 = g.get_overlaps(read, sin)
            assert n1 == n2, ("overlap count", i, n1, n2)
            if n1 > 0:
                assert (o1 == o2).all(), ("overlaps", i)
                assert (s1 == s2).all(), ("similarity", i)   # IEEE doubles, bit-equal
            assert r.index_checksum() == g.index_checksum(), ("index", i)
            checks += 1
        if t[0] == "C":
            g = api.SeqSet(int(t[1]), lib)
            r = ref.RefSeqSet(int(t[1]))
        elif t[0] == "O":
            break
        else:
            tr.replay([t], lambda k: None) if False else None
            _apply(t, r)
            _apply(t, g)
    assert checks > 5


def _apply(t, s):
    c = t[0]
    if c == "A":
        s.add_read(t[1], "" if t[2] == "." else t[2], int(t[3]), int(t[4]), int(t[5]), int(t[6]), float(t[7]))
    elif c == "R":
        s.repeat_add_read(t[1])
    elif c == "N":
        s.input_novel_read(t[1], t[2], int(t[3]), int(t[4]))
    elif c == "U":
        s.update_all_consensus()
    elif c == "K":
        s.change_kmer_length(int(t[1]))
    elif c == "H":
        s.set_hit_len_required(int(t[1]))


def dp_cases(seed, n=300):
    """Random GlobalAlignment_PosWeight problems: equal and unequal lengths, clean / noisy / indel inputs."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        lent = int(rng.integers(0, 70))
        kind = rng.integers(0, 5)
        t = rng.integers(0, 4, size=lent)
        p = list(t)
        if kind == 0:
            pass
        elif kind == 1:                      # substitutions
            for _ in range(int(rng.integers(1, 6))):
                if p:
                    p[int(rng.integers(len(p)))] = int(rng.integers(4))
        elif kind == 2:                      # an indel
            if len(p) > 3:
                x = int(rng.integers(1, len(p) - 1))
                if rng.random() < 0.5:
                    del p[x]
                else:
                    p.insert(x, int(rng.integers(4)))
        elif kind == 3:                      # unrelated, maybe other length
            p = list(rng.integers(0, 4, size=max(0, lent + int(rng.integers(-4, 5)))))
        else:                                # indel + substitutions, N's
            if len(p) > 6:
                x = int(rng.integers(2, len(p) - 2))
                del p[x:x + int(rng.integers(1, 3))]
                p[int(rng.integers(len(p)))] = 4
        tw = np.zeros((lent, 4), dtype=np.int32)
        for j in range(lent):
            tw[j, t[j]] = int(rng.integers(1, 30))
            if rng.random() < 0.3:
                tw[j, int(rng.integers(4))] += int(rng.integers(0, 12))
            if rng.random() < 0.03:
                tw[j] = 0
        ps = "".join("ACGTN"[c] for c in p)
        out.append((tw, ps))
    return out


def check_dp(lib, ref, seed=5):
    cases = dp_cases(seed)
    got = api.dp_pos_weight_batch(cases, lib)
    for (tw, p), (sc, ed) in zip(cases, got):
        rs, re_ = ref.dp_pos_weight(tw, p)
        assert (sc, ed) == (rs, re_), (tw.tolist(), p, sc, rs, ed, re_)


def dp_equal_cases(seed=11, n=260):
    """Equal-length GlobalAlignment_PosWeight problems as the hot path poses them (overhangs, same-diagonal gaps):
    clean, substitution bursts, frame shifts that an in-band gap pair can repair, N's, mixed-support columns,
    lengths on both sides of the shared-memory limit of the half-warp DP (192)."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        L = int(rng.choice([2, 3, 7, 12, 13, 14, 30, 45, 64, 100, 150, 191, 192, 230, 300])) if i % 3 == 0 else int(rng.integers(2, 160))
        t = rng.integers(0, 4, size=L)
        p = list(t)
        kind = int(rng.integers(0, 6))
        if kind == 1:
            for _ in range(int(rng.integers(1, 4))):
                p[int(rng.integers(L))] = int(rng.integers(4))
        elif kind == 2:                      # > 2 substitutions: forces the banded DP, answer stays on the diagonal
            for _ in range(int(rng.integers(3, 9))):
                x = int(rng.integers(L))
                p[x] = (p[x] + 1 + int(rng.integers(3))) % 4
        elif kind == 3 and L > 12:           # delete d bases early, insert d later: a frame shift inside the band
            d = int(rng.integers(1, 5))
            x = int(rng.integers(1, L - d - 4))
            del p[x:x + d]
            y = int(rng.integers(x + 1, len(p)))
            for _ in range(d):
                p.insert(y, int(rng.integers(4)))
        elif kind == 4:                      # unrelated
            p = list(rng.integers(0, 4, size=L))
        elif kind == 5:                      # N's + substitutions
            for _ in range(int(rng.integers(1, 4))):
                p[int(rng.integers(L))] = 4
            for _ in range(int(rng.integers(0, 6))):
                p[int(rng.integers(L))] = int(rng.integers(4))
        assert len(p) == L
        tw = np.zeros((L, 4), dtype=np.int32)
        for j in range(L):
            tw[j, t[j]] = int(rng.integers(1, 30))
            if rng.random() < 0.3:
                tw[j, int(rng.integers(4))] += int(rng.integers(0, 12))
            if rng.random() < 0.03:
                tw[j] = 0
        out.append((tw, "".join("ACGTN"[c] for c in p)))
    return out


def _diag_mismatches(tw, p):
    """Mismatches of the all-diagonal alignment under AlignAlgo::IsBaseEqual (AlignAlgo.hpp:49-55)."""
    x = 0
    for j, c in enumerate(p):
        s = int(tw[j].sum())
        if s == 0 or c == "N":
            continue
        if not s < 3 * int(tw[j, "ACGT".index(c)]):
            x += 1
    return x


def check_dp_hot(lib, ref, seed, variant):
    """The DP routines the stream kernel really runs, against AlignAlgo::GlobalAlignment_PosWeight (AlignAlgo.hpp:57-216):
    score and edit string.  variant 0 = t4_dp_equal (has the reference's <= 2-mismatch fast path), variant 1 =
    w_dp_equal_half (always the banded DP; its caller only invokes it beyond 2 mismatches, so only those cases count)."""
    cases = dp_equal_cases(seed)
    if variant == 1:
        cases = [(tw, p) for tw, p in cases if _diag_mismatches(tw, p) > 2]
        assert len(cases) > 40
    got = api.dp_hot_path_batch(cases, variant, lib)
    for (tw, p), (sc, ed) in zip(cases, got):
        rs, re_ = ref.dp_pos_weight(tw, p)
        assert (sc, ed) == (rs, re_), (variant, len(p), p, sc, rs, ed, re_)


def check_big_repeats(lib, ref, n_copies=10050):
    """A k-mer with more than 10000 postings: the `repeats > 10000` rules of GetOverlapsFromHits, including the
    run-local `hits[k]` indexing slip (SeqSet.hpp:931-947), and the >=100-postings skip rule of GetHitsFromRead."""
    lib.check(lib.reset())
    rng = np.random.default_rng(77)
    base = "".join("ACGT"[c] for c in rng.integers(0, 4, size=120))
    other = "".join("ACGT"[c] for c in rng.integers(0, 4, size=150))
    g = api.SeqSet(9, lib)
    r = ref.RefSeqSet(9)
    # many contigs that all carry the k-mers of `base`; each gets a unique tail so they stay distinct sequences
    tails = ["".join("ACGT"[c] for c in rng.integers(0, 4, size=30)) for _ in range(64)]
    reads = [base + tails[i % 64] for i in range(n_copies)]
    for rd in reads:
        r.input_novel_read("IGHV1-2*01", rd, 1, -1)
        g.input_novel_read("IGHV1-2*01", rd, 1, -1)
    assert g.size() == r.size() == n_copies
    assert g.index_checksum() == r.index_checksum()
    for q in (base[10:110] + other[:50], other[:60] + base[:90], base[:100], other):
        for strand in (0, 1):
            hr = canon_hits(r.get_hits(q, strand))
            hg = g.get_hits(q, strand)
            assert hr.shape == hg.shape and (hr == hg).all()
            if q is not other:
                assert hg[:, 4].max() > 10000      # the scenario really has a k-mer with > 10000 postings (hg equals hr)
            n1, o1, s1 = r.get_overlaps(q, strand)
            n2, o2, s2 = g.get_overlaps(q, strand)
            assert n1 == n2, (n1, n2)
            if n1 > 0:
                assert (o1 == o2).all() and (s1 == s2).all()
        assert g.add_read(q, "IGHV", 0, -1, 1, 0, 0.9) == r.add_read(q, "IGHV", 0, -1, 1, 0, 0.9)
    assert g.index_checksum() == r.index_checksum()
    # the batch probe on the same set: lists of > 10000 postings (streamed, `repeats > 10000` flag), the >= 100 rules
    qs = [base[10:110] + other[:50], other[:60] + base[:90], base[:100], other, base + other + base[:60]]
    d = np.zeros(2 * len(qs), dtype=synth.READ_DESC)
    o = 0
    for i, q in enumerate(qs + qs):
        d[i]["seq_off"], d[i]["len"], d[i]["barcode"], d[i]["strand_in"] = o, len(q), -1, 0 if i < len(qs) else 1
        o += len(q)
    pool = np.frombuffer(("".join(qs + qs) + "\0" * 16).encode(), dtype=np.uint8).copy()
    wl = api.Workload(d, pool, [], lib)
    hits = api.Hits(len(d), 24 << 20, lib)
    for skip in (0, 1):
        api.streams_get_hits([g], wl, [0, len(d)], hits, allow_total_skip=skip)
        assert hits.stats()["records"] == len(d)       # also raises when the key buffer was too small
        for i, q in enumerate(qs + qs):
            hr = _canon4(r.get_hits(q, int(d[i]["strand_in"]), -1, bool(skip)))
            hg, fl = hits.fetch(i)
            hg = _canon4(hg)
            assert hr.shape == hg.shape and (hr == hg).all(), ("big probe", i, skip)
            if skip == 0 and q is not other:
                assert fl & 1
    wl.close()
    hits.close()


def check_barcode_mode(lib, ref, seed=31, n_barcodes=5):
    """Barcode mode inside one stream (BASELINE configs[3] flavour): barcode-salted index keys
    (KmerIndex.hpp:29-33), per-hit barcode filter and repeats = 1 (SeqSet.hpp:1394-1418), hitLenRequired 13,
    ExtendOverlap mismatch factor 2.0, no periodic consensus update (main.cpp:1549-1560, 1862).
    ReleaseFinishedBarcodeSeq is not part of this path (both sides skip it)."""
    lib.check(lib.reset())
    w = small_workload(seed, 20, 500)
    d = w.descs.copy()
    L = w.L
    reads = w.pool.reshape(-1, L)
    h = (reads.astype(np.int64) * np.arange(1, L + 1)).sum(axis=1)
    d["barcode"] = (h % n_barcodes).astype(np.int32)
    d["sim_threshold"] = 0.9
    d["mate_idx"] = -1
    cfg = synth.run_cfg(has_barcode=1)
    g = api.SeqSet(9, lib)
    r = ref.RefSeqSet(9)
    for s in (g, r):
        s.set_hit_len_required(13)
    g.set_consider_barcode_in_hash(1)
    r.set_consider_barcode_in_hash(1)
    _, gret, gstr, gres = g.run_descs(cfg, d, w.pool, w.names)
    _, rret, rstr, rres = r.run_descs(cfg, d, w.pool, w.names)
    assert (gret == rret).all() and (gstr == rstr).all() and (gres == rres).all()
    assert g.output() == r.output()
    assert g.index_checksum() == r.index_checksum()
    assert len(set(c["barcode"] for c in (g.get_contig(i) for i in range(g.size())) if c)) > 1


def _barcode_descs(seed, n_barcodes=3, nclones=6, npairs=400):
    """A barcode-sorted record list (main.cpp:1126 CompReadWithBarcode order) over a small synthetic library."""
    cl = synth.make_clones(nclones, seed)
    rd = synth.sample_pairs(cl, npairs, 150, seed)
    w = synth.build_workload(cl, rd)
    d = w.descs.copy()
    reads = w.pool.reshape(-1, w.L)
    h = (reads.astype(np.int64) * np.arange(1, w.L + 1)).sum(axis=1) % n_barcodes
    order = np.argsort(h, kind="stable")
    d = d[order]
    d["barcode"] = h[order].astype(np.int32)
    d["mate_idx"] = -1
    d["sim_threshold"] = 0.9
    n = len(d)
    same_prev = np.zeros(n, dtype=bool)
    rs = reads[order]
    same_prev[1:] = (rs[1:] == rs[:-1]).all(axis=1) & (d["barcode"][1:] == d["barcode"][:-1])
    d["flags"] = np.where(same_prev, d["flags"] | synth.RD_DUP, d["flags"] & ~np.uint32(synth.RD_DUP))
    d["eq_lo"] = np.arange(n)
    d["eq_hi"] = np.arange(n) + 1
    return w, d


def _same_sets(g, r):
    assert g.size() == r.size()
    assert g.output() == r.output()
    assert g.index_checksum() == r.index_checksum()
    for i in range(g.size()):
        gc = g.get_contig(i)
        assert (gc is None) == (r.num_read(i) < 0), i
        if gc is not None:
            assert gc["num_read"] == r.num_read(i), i


def check_barcode_release(lib, ref, seed=33):
    """SeqSet::ReleaseFinishedBarcodeSeq (SeqSet.hpp:10815; driver main.cpp:1846-1859: only reads with addRet >= 0 count
    towards "finished"), ReleaseShallowContigs (SeqSet.hpp:10928) and IsContigShallow (:2512): inside the batch loop
    (cfg.release_barcodes, contig_min_cov 0 / 2 / 20) and through the per-call entries, against the reference --
    Output text, slot count, numRead of every slot and the index multiset (purged contigs leave the index)."""
    w, d = _barcode_descs(seed)
    base_sum = None
    for min_cov in (0, 2, 20):
        lib.check(lib.reset())
        outs = []
        for release in (0, 1):
            cfg = synth.run_cfg(has_barcode=1, release_barcodes=release, contig_min_cov=min_cov)
            r = ref.RefSeqSet(9)
            r.set_hit_len_required(13)
            r.set_consider_barcode_in_hash(1)
            _, rret, rstr, rres = r.run_descs(cfg, d, w.pool, w.names)
            g = api.SeqSet(9, lib)
            g.set_hit_len_required(13)
            g.set_consider_barcode_in_hash(1)
            _, gret, gstr, gres = g.run_descs(cfg, d, w.pool, w.names)
            assert (gret == rret).all() and (gstr == rstr).all() and (gres == rres).all()
            _same_sets(g, r)
            outs.append((r.output(), r.index_checksum()[0]))
            if release == 1 and min_cov > 0:
                # --contigMinCov: the driver's last step before Output (main.cpp:1952-1955)
                r.release_shallow_contigs(min_cov)
                g.release_shallow_contigs(min_cov)
                assert g.output() == r.output()
                assert g.size() == r.size()
                outs.append((r.output(), 0))
        if min_cov == 0:
            assert outs[1][1] < outs[0][1]       # the purge really happened: postings left the index ...
            assert outs[0][0] == outs[1][0]      # ... and is invisible in Output when nothing is shallow
            assert len(outs[0][0]) > 1000
        if min_cov == 20:
            assert 0 < len(outs[1][0]) < len(outs[0][0])    # shallow contigs were dropped inside the loop, deep ones stayed
    # per-call route, like the driver: assemble one barcode, purge it (the purge walks the slots from the end and stops at
    # the first contig of another barcode or an already purged one), go on with the next
    lib.check(lib.reset())
    cfg = synth.run_cfg(has_barcode=1, final_update=0, do_rescue=0)
    r = ref.RefSeqSet(9)
    r.set_hit_len_required(13)
    r.set_consider_barcode_in_hash(1)
    g = api.SeqSet(9, lib)
    g.set_hit_len_required(13)
    g.set_consider_barcode_in_hash(1)
    for bc, cov in ((0, 0), (1, 20), (2, 2)):
        part = d[d["barcode"] == bc].copy()
        part["flags"][0] &= ~np.uint32(synth.RD_DUP)
        _, rret, _, _ = r.run_descs(cfg, part, w.pool, w.names)
        _, gret, _, _ = g.run_descs(cfg, part, w.pool, w.names)
        assert (gret == rret).all()
        if bc == 2:
            r.release_finished_barcode(1, 0)     # stops at once: the tail belongs to barcode 2
            g.release_finished_barcode(1, 0)
            _same_sets(g, r)
        r.release_finished_barcode(bc, cov)
        g.release_finished_barcode(bc, cov)
        _same_sets(g, r)
    purged = [g.contig_flags(i) for i in range(g.size())]
    assert 1 in purged and -1 in purged      # purged contigs and (barcode 1, cov 20) dropped ones
    # a purged set survives UpdateAllConsensus and ChangeKmerLength (Clean skips contigs with index == false)
    r.update_all_consensus()
    g.update_all_consensus()
    _same_sets(g, r)


def check_single_cell(lib, ref, seed=51, n_barcodes=24, reads_per_barcode=150, n_shards=5, contig_min_cov=0):
    """BASELINE configs[3] in small: 10x-style barcoded single-end reads, whole barcodes per stream (SURVEY.md 8e),
    hitLenRequired 13, barcode-salted index, finished barcodes purged -- per stream against the reference SeqSet driven
    by the restated loop (return codes, strands, rescue codes, Output with barcode slots, index multiset, numRead)."""
    lib.check(lib.reset())
    cl = synth.make_clones(60, seed)
    rd, bc = synth.sample_single_cell(cl, n_barcodes, reads_per_barcode, 150, seed)
    w = synth.build_workload(cl, rd, barcode=bc)
    cfg = synth.run_cfg(has_barcode=1, release_barcodes=1, contig_min_cov=contig_min_cov)
    off, descs = synth.shard_workload(w, n_shards, align="barcode")
    for j in range(1, n_shards):     # no barcode straddles two streams
        assert descs["barcode"][off[j] - 1] != descs["barcode"][off[j]]
    sets = api.SeqSet.create_many(n_shards, 9, lib, hit_len_required=13, consider_barcode=1)
    ret, strands, resc = api.streams_run(sets, cfg, descs, off, w.pool, w.names, lib)
    total = 0
    for j in range(n_shards):
        lo, hi = int(off[j]), int(off[j + 1])
        r = ref.RefSeqSet(9)
        r.set_hit_len_required(13)
        r.set_consider_barcode_in_hash(1)
        _, rret, rstr, rresc = r.run_descs(cfg, descs[lo:hi].copy(), w.pool, w.names)
        assert (rret == ret[lo:hi]).all(), ("ret", j, np.flatnonzero(rret != ret[lo:hi])[:5])
        assert (rstr == strands[lo:hi]).all() and (rresc == resc[lo:hi]).all(), ("strand/rescue", j)
        _same_sets(sets[j], r)
        total += int((rret >= 0).sum())
    assert total > n_barcodes * reads_per_barcode // 2
    return total


def check_repseq(lib, ref, seed=61, n_reads=4000, n_shards=3):
    """BASELINE configs[4] in small: --repseq (trimLevel 2) amplicon TCR-seq reads, 100 bp single end: repetitiveData = true
    (skip-repeats first pass SeqSet.hpp:1520-1531, ExtendOverlap mismatch factor 2.0 :1226-1237), V-gene pseudo barcodes
    on an unsalted index (main.cpp:1224-1235), halved k-change threshold (main.cpp:1567)."""
    lib.check(lib.reset())
    cl = synth.make_clones(120, seed, chains=("TRB",))
    rd = synth.sample_amplicon(cl, n_reads, 100, seed)
    w = synth.build_workload(cl, rd, repseq=True)
    assert (w.descs["barcode"] >= 0).mean() > 0.5
    cfg = synth.run_cfg(repetitive=1, change_k_threshold=40, first_read_len=100)      # small threshold: k changes mid-run
    off, descs = synth.shard_workload(w, n_shards)
    sets = api.SeqSet.create_many(n_shards, 9, lib, hit_len_required=50)           # main.cpp:1541-1547: max(21, L/2) when L/2 < 31 -> here L/2 = 50 > 31 keeps 31; exercise the setter anyway
    for s_ in sets:
        s_.set_hit_len_required(31)
    ret, strands, resc = api.streams_run(sets, cfg, descs, off, w.pool, w.names, lib)
    for j in range(n_shards):
        lo, hi = int(off[j]), int(off[j + 1])
        r = ref.RefSeqSet(9)
        _, rret, rstr, rresc = r.run_descs(cfg, descs[lo:hi].copy(), w.pool, w.names)
        assert (rret == ret[lo:hi]).all(), ("ret", j, np.flatnonzero(rret != ret[lo:hi])[:5])
        assert (rstr == strands[lo:hi]).all() and (rresc == resc[lo:hi]).all(), ("strand/rescue", j)
        assert r.output() == sets[j].output(), ("contigs", j)
        assert r.index_checksum() == sets[j].index_checksum(), ("index", j)
        assert r.kmer_length() == sets[j].kmer_length()
    assert int((ret >= 0).sum()) > n_reads // 2


def check_dup_runs(lib, ref, seed=71):
    """Long runs of duplicate records (amplicon data: every read of a clonotype is the same string): the device applies a
    run of RepeatAddRead calls in one pass; the periodic UpdateAllConsensus (here every 37 assembled reads) and a pending
    k change must still see exactly the reference's state."""
    lib.check(lib.reset())
    cl = synth.make_clones(7, seed, chains=("TRB",))
    rd = synth.sample_amplicon(cl, 6000, 100, seed, alpha=0.7, sub_rate=0.001)
    w = synth.build_workload(cl, rd, repseq=True)
    assert (w.descs["flags"] & synth.RD_DUP).mean() > 0.8
    for every, chk in ((37, 4096), (10000, 3), (5000, 4096)):
        lib.check(lib.reset())
        cfg = synth.run_cfg(repetitive=1, change_k_threshold=chk, update_consensus_every=every, first_read_len=100)
        g = api.SeqSet(9, lib)
        r = ref.RefSeqSet(9)
        _, gret, gstr, gres = g.run_descs(cfg, w.descs, w.pool, w.names)
        _, rret, rstr, rres = r.run_descs(cfg, w.descs, w.pool, w.names)
        assert (gret == rret).all() and (gstr == rstr).all() and (gres == rres).all(), (every, chk)
        assert g.output() == r.output(), (every, chk)
        assert g.index_checksum() == r.index_checksum() and g.kmer_length() == r.kmer_length()
        for i in range(g.size()):
            c = g.get_contig(i)
            assert (c is None) == (r.num_read(i) < 0) and (c is None or c["num_read"] == r.num_read(i))


def check_input_novel_fa(lib, ref, tmp_path):
    """SeqSet::InputNovelFa (SeqSet.hpp:2986, --debug-ns)."""
    lib.check(lib.reset())
    rng = np.random.default_rng(3)
    fa = tmp_path / "ns.fa"
    with open(fa, "w") as f:
        for i in range(7):
            s = "".join("ACGT"[c] for c in rng.integers(0, 4, size=int(rng.integers(40, 400))))
            f.write(">ns%d some comment\n" % i)
            for j in range(0, len(s), 60):
                f.write(s[j:j + 60] + "\n")
    r = ref.RefSeqSet(9)
    g = api.SeqSet(9, lib)
    r.input_novel_fa(str(fa))
    assert g.input_novel_fa(str(fa)) == 7
    assert g.output() == r.output() and len(g.output()) > 500
    assert g.index_checksum() == r.index_checksum()


def _run_resident(lib, sets, cfg, wl, off):
    hs = (api.C.c_void_p * len(sets))(*[s.h for s in sets])
    off = np.ascontiguousarray(off, dtype=np.int64)
    lib.check(lib.streams_run_resident(hs, len(sets), cfg.ctypes.data, wl.h, off.ctypes.data, None))
    n = wl.n
    ret = np.zeros(n, dtype=np.int32)
    strands = np.zeros(n, dtype=np.int8)
    resc = np.zeros(n, dtype=np.int32)
    lib.check(lib.workload_results(wl.h, ret.ctypes.data, strands.ctypes.data, resc.ctypes.data))
    return ret, strands, resc


def check_assign_pass(lib, ref, seed, n_shards, nclones=25, npairs=400, kmer=17, group="", workload=None, cfg=None, n_workers=0,
                      drop=0.0):
    """t4_streams_assign_reads (SURVEY.md 8f-2) against the reference's own pass (main.cpp:2047-2118): for every shard the
    extended set built by InputSeqSet at k, AssignRead of every assembled read in the driver's order (identical
    neighbours share a call) with novelSeqSimilarity 0.95, and RecomputePosWeight -- per read the assigned contig,
    coordinates, strand, matchCnt and the similarity double; per extended set the Output text (consensus + recomputed
    posWeight) and the index checksum."""
    lib.check(lib.reset())
    w = workload if workload is not None else small_workload(seed, nclones, npairs)
    cfg = cfg if cfg is not None else synth.run_cfg()
    off, descs = synth.shard_workload(w, n_shards, balance="cost" if group else "reads", group=group)
    n_shards = len(off) - 1
    if drop > 0:   # reads the driver's gene-order / constant-gene filters reject (main.cpp:1609-1654): never assembled, never listed
        descs = descs.copy()
        rng = np.random.default_rng(seed)
        descs["flags"] |= np.where(rng.random(len(descs)) < drop, synth.RD_FILTERED, 0).astype(descs["flags"].dtype)
    sets = api.SeqSet.create_many(n_shards, 9, lib)
    wl = api.Workload(descs, w.pool, w.names, lib)
    ret, strands, resc = _run_resident(lib, sets, cfg, wl, off)
    a = api.Assign(sets, wl, off, kmer, n_workers=n_workers)
    ga, gs = a.results()
    st = a.stats()
    n_listed = n_assigned = n_calls = 0
    for j in range(n_shards):
        lo, hi = int(off[j]), int(off[j + 1])
        r = ref.RefSeqSet(9)
        d = descs[lo:hi].copy()
        _, rret, rstr, rresc = r.run_descs(cfg, d, w.pool, w.names)
        assert (rret == ret[lo:hi]).all() and (rstr == strands[lo:hi]).all() and (rresc == resc[lo:hi]).all(), ("assembly", j)
        lst = ref.assembled_list(rret, rresc)
        ext, ra, rs = ref.assign_pass(r, kmer, d, w.pool, lst, rstr)
        listed = np.zeros(hi - lo, dtype=bool)
        listed[lst] = True
        assert (ga[lo:hi][~listed, 0] == api.ASSIGN_NOT_LISTED).all(), ("not listed", j)
        g = ga[lo:hi][lst]
        assert (g[:, 0] == ra[:, 0]).all(), ("seqIdx", j, np.flatnonzero(g[:, 0] != ra[:, 0])[:5])
        ok = ra[:, 0] >= 0
        assert (g[ok] == ra[ok]).all(), ("overlap", j, np.flatnonzero((g[ok] != ra[ok]).any(axis=1))[:5])
        assert (gs[lo:hi][lst][ok] == rs[ok]).all(), ("similarity", j)
        ge = a.extended_set(j)
        assert ge.kmer_length() == kmer and ge.size() == ext.size()
        assert ge.output() == ext.output(), ("extended set", j)
        assert ge.index_checksum() == ext.index_checksum(), ("extended index", j)
        n_listed += len(lst)
        n_assigned += int(ok.sum())
        rd = [bytes(w.pool[int(x["seq_off"]):int(x["seq_off"]) + int(x["len"])]) for x in d[lst]]
        n_calls += sum(1 for i in range(len(rd)) if i == 0 or rd[i] != rd[i - 1])
    assert st["reads"] == n_listed and st["assigned"] == n_assigned and st["assign_calls"] == n_calls, (st, n_listed, n_assigned, n_calls)
    a.close()
    wl.close()
    return n_listed, n_assigned


def check_kmer_count_stats(lib, ref, seed=101, n=1500, k=21):
    """t4_kmer_count_stats (SURVEY.md 8f-3) against the reference's KmerCount: AddCount of every read, then
    GetCountStatsAndTrim without trimming -- min / median exact, avg the same float.  Reads: sampled pairs of a clone set
    (shared k-mers with high counts) plus ragged ones: lengths 5..400, N's, reads of N's only, homopolymers, duplicates."""
    rng = np.random.default_rng(seed)
    cl = synth.make_clones(30, seed)
    rd = synth.sample_pairs(cl, n // 3, 150, seed, sub_rate=0.01)
    reads = [synth.decode(c) for c in rd.codes]
    src = reads[: 50]
    while len(reads) < n:
        s = src[int(rng.integers(len(src)))]
        L = int(rng.integers(5, 401))
        t = (s * 4)[int(rng.integers(0, 100)):][:L]
        kind = int(rng.integers(0, 8))
        if kind == 0:
            t = "N" * L
        elif kind == 1:
            t = "ACGT"[int(rng.integers(4))] * L
        elif kind in (2, 3):
            t = list(t)
            for p in rng.integers(0, L, size=int(rng.integers(1, 6))):
                t[int(p)] = "N"
            t = "".join(t)
        elif kind == 4 and len(reads) > 3:
            t = reads[int(rng.integers(len(reads)))]
        reads.append(t)
    lens = np.array([len(r) for r in reads], dtype=np.int32)
    off = np.zeros(len(reads), dtype=np.uint64)
    off[1:] = np.cumsum(lens[:-1])
    pool = np.frombuffer(("".join(reads) + "\0" * 16).encode(), dtype=np.uint8).copy()
    # qualities: mostly good; a third of the N-free reads get a bad tail (Phred <= 15 from some position on, some sparse,
    # some whole reads) so that the trimming rules fire: cut positions, reads cut below k (dropped), untouched reads
    quals = []
    for t in reads:
        q = ["I"] * len(t)
        if "N" not in t and len(t) > 30 and rng.random() < 0.35:
            mode = int(rng.integers(0, 4))
            st = int(rng.integers(0, len(t))) if mode != 3 else 0
            for p in range(st, len(t)):
                if mode == 1 and rng.random() < 0.5:
                    continue
                q[p] = "#$%&'()*+,-./0"[int(rng.integers(0, 14))]     # Phred 2..15
            if mode == 2:
                q[-1] = "I"
        quals.append("".join(q))
    qpool = np.frombuffer(("".join(quals) + "\0" * 16).encode(), dtype=np.uint8).copy()
    n_trim = 0
    for qp in (None, qpool):
        rmn, rmed, ravg, rnl = ref.kmer_count_stats(pool, off, lens, k, qual=qp)
        gmn, gmed, gavg, gnl = api.kmer_count_stats(pool, off, lens, k, lib, qual=qp)
        assert (gnl == rnl).all(), ("new length", qp is not None, np.flatnonzero(gnl != rnl)[:5])
        assert (gmn == rmn).all(), ("min", qp is not None, np.flatnonzero(gmn != rmn)[:5])
        assert (gmed == rmed).all(), ("median", qp is not None, np.flatnonzero(gmed != rmed)[:5])
        assert (gavg.view(np.uint32) == ravg.view(np.uint32)).all(), ("avg", qp is not None, np.flatnonzero(gavg.view(np.uint32) != ravg.view(np.uint32))[:5])
        if qp is None:
            assert (rnl == lens).all()
            assert (rmn < 0).sum() > 10 and (rmn == 0).sum() > 10 and (rmn > 1).sum() > 100 and rmed.max() > 20
        else:
            n_trim = int((rnl < lens).sum())
            assert n_trim > 50 and ((rnl == 0) & (lens >= k)).sum() > 3
    return int(len(reads))


def write_gene_fasta(path, messy=True):
    """The bundled gene pool as FASTA; `messy` adds what InputRefFa has to clean up: IMGT '.' gaps, lower case, ambiguity
    codes, a duplicated sequence under another name, the same record twice, a '/OR' pseudo-gene, multi-line records."""
    pool = synth.load_gene_pool()
    recs = []
    for ch in pool.values():
        for seg in ch.values():
            for name, seq in seg:
                recs.append((name, seq))
    out = []
    for i, (name, seq) in enumerate(recs):
        s = seq
        if messy and i % 7 == 0:
            s = s[:30] + "..." + s[30:60] + "......" + s[60:]
        if messy and i % 11 == 0 and len(s) > 80:
            s = s[:70] + s[70:75].lower() + s[75:]
        if messy and i % 13 == 0 and len(s) > 90:
            s = s[:85] + "RY" + s[87:]
        out.append((name, s))
    if messy:
        out.insert(5, ("IGHV9-99*01 extra words", recs[2][1]))                 # same sequence as another gene: names joined
        out.insert(9, (recs[3][0], recs[3][1]))                                 # the same record again: dropped
        out.insert(12, ("IGHV3/OR16-9*01", recs[20][1][:200] + "ACGTACGTTTGACCA"))  # /OR pseudo-gene: skipped
        out.insert(14, ("TRBD1*01", "GGGACAGGGGGC"))                            # D genes are kept (short: below k + a few)
    with open(path, "w") as f:
        for name, s in out:
            f.write(">%s\n" % name)
            for p in range(0, len(s), 60):
                f.write(s[p:p + 60] + "\n")
    return recs


def check_refset_scan(lib, ref, tmp_path, seed=121, n=1200, radius=None, hit_len=27, k=9):
    """t4_refset_create_from_fa + t4_refset_scan (SURVEY.md 8f-4) against the reference: InputRefFa (kept sequences, joined
    names, the k-mer index) and, per read, IsLowComplexity and HasHitInSet(read, 0) -- candidate reads from clonotypes on both
    strands, random reads, chimeras of a gene piece and random sequence, reads with N's, low-complexity reads, short reads,
    reads with indels against the gene (several diagonals inside the radius)."""
    rng = np.random.default_rng(seed)
    fa = os.path.join(str(tmp_path), "genes_%d.fa" % seed)
    recs = write_gene_fasta(fa)
    lib.check(lib.reset())
    g = api.RefSet(fa, k, lib, hit_len_required=hit_len)
    r = ref.RefGeneSet(fa, k, hit_len_required=hit_len)
    if radius is not None:
        g.set_radius(radius)
        r.set_radius(radius)
    assert g.names() == r.names() and g.size() > 100
    assert g.seqset().index_checksum() == r.index_checksum()
    cl = synth.make_clones(40, seed)
    rd = synth.sample_pairs(cl, 200, 150, seed, sub_rate=0.02)
    reads = [synth.decode(c) for c in rd.codes]
    comp = {"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}
    genes = [s for _, s in recs if len(s) > 200]

    def rnd(L):
        return "".join("ACGT"[c] for c in rng.integers(0, 4, size=L))

    while len(reads) < n:
        kind = int(rng.integers(0, 10))
        L = int(rng.integers(20, 260))
        gs = genes[int(rng.integers(len(genes)))]
        p = int(rng.integers(0, max(1, len(gs) - 60)))
        piece = gs[p:p + L]
        if kind == 0:
            t = rnd(L)
        elif kind == 1:
            t = piece[: max(10, len(piece) // 3)] + rnd(L)
        elif kind == 2:
            t = rnd(L // 2) + piece[: 20 + int(rng.integers(0, 40))] + rnd(L // 3)
        elif kind == 3:
            t = "".join(comp[c] for c in reversed(piece))
        elif kind == 4:
            t = list(piece)
            for q in rng.integers(0, max(1, len(t)), size=int(rng.integers(1, 8))):
                t[int(q)] = "N"
            t = "".join(t)
        elif kind == 5:
            t = "ACGT"[int(rng.integers(4))] * (L // 2) + piece[: L // 3]
        elif kind == 6:     # indels: deletions / insertions of 1-6 bases move the chain across neighbouring diagonals
            t = piece
            for _ in range(int(rng.integers(1, 4))):
                q = int(rng.integers(5, max(6, len(t) - 5)))
                d = int(rng.integers(1, 7))
                t = t[:q] + (rnd(d) if rng.random() < 0.5 else "") + t[q + (d if rng.random() < 0.5 else 0):]
        elif kind == 7:
            t = piece[: int(rng.integers(5, 30))]
        elif kind == 8:     # two genes in one read
            g2 = genes[int(rng.integers(len(genes)))]
            t = piece[: L // 2] + g2[-(L // 2):]
        else:
            t = piece
        if len(t) < 1:
            t = "A"
        reads.append(t[:400])
    lens = np.array([len(x) for x in reads], dtype=np.int32)
    off = np.zeros(len(reads), dtype=np.uint64)
    off[1:] = np.cumsum(lens[:-1])
    pool = np.frombuffer(("".join(reads) + "\0" * 16).encode(), dtype=np.uint8).copy()
    gs_, gl_, st = g.scan(pool, off, lens)
    rs_ = np.array([r.has_hit_in_set(x, 0) for x in reads], dtype=np.int8)
    rl_ = np.array([ref.is_low_complexity(x) for x in reads], dtype=np.uint8)
    assert (gl_ == rl_).all(), ("low complexity", np.flatnonzero(gl_ != rl_)[:5])
    assert (gs_ == rs_).all(), ("HasHitInSet", np.flatnonzero(gs_ != rs_)[:8], gs_[gs_ != rs_][:8], rs_[gs_ != rs_][:8])
    assert st["with_hit"] == int((rs_ != 0).sum()) and st["low_complexity"] == int(rl_.sum())
    assert (rs_ == 1).sum() > 50 and (rs_ == -1).sum() > 50 and (rs_ == 0).sum() > 50 and rl_.sum() > 10
    g.close()
    return int((rs_ != 0).sum())


def check_refset_overlaps(lib, ref, tmp_path, seed=131, n=500, radius=None, hit_len=31, k=9):
    """t4_refset_get_overlaps against SeqSet::GetOverlapsFromRead(read, 0, -1, 0, false) on the reference's gene set (the call
    AnnotateRead makes per read): every overlap's gene, coordinates, strand, matchCnt, indelCnt and the similarity double,
    in order.  Reads: clonotype reads (V + junction + J + C: several genes per read), gene pieces with substitutions and
    indels (gaps scored by the affine GlobalAlignment), chimeras, reverse strands, short V-end / J-start reads (the
    GetVJOverlapsFromHits rescue), random reads."""
    rng = np.random.default_rng(seed)
    fa = os.path.join(str(tmp_path), "genes_o%d.fa" % seed)
    recs = write_gene_fasta(fa)
    lib.check(lib.reset())
    g = api.RefSet(fa, k, lib, hit_len_required=hit_len)
    r = ref.RefGeneSet(fa, k, hit_len_required=hit_len)
    if radius is not None:
        g.set_radius(radius)
        r.set_radius(radius)
    cl = synth.make_clones(30, seed)
    rd = synth.sample_pairs(cl, n // 4, 150, seed, sub_rate=0.02)
    reads = [synth.decode(c) for c in rd.codes]
    comp = {"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}
    byname = dict(recs)
    vjs_v = [(nm, s) for nm, s in recs if len(nm) > 3 and nm[3] == "V" and len(s) > 250]
    vjs_j = [(nm, s) for nm, s in recs if len(nm) > 3 and nm[3] == "J" and len(s) > 35]
    genes = [s for _, s in recs if len(s) > 200]

    def rnd(L):
        return "".join("ACGT"[c] for c in rng.integers(0, 4, size=L))

    def mutate(t, subs, indels):
        t = list(t)
        for _ in range(subs):
            q = int(rng.integers(0, len(t)))
            t[q] = "ACGT"[int(rng.integers(4))]
        t = "".join(t)
        for _ in range(indels):
            q = int(rng.integers(12, max(13, len(t) - 12)))
            d = int(rng.integers(1, 5))
            t = t[:q] + (rnd(d) if rng.random() < 0.5 else "") + t[q + (d if rng.random() < 0.5 else 0):]
        return t

    while len(reads) < n:
        kind = int(rng.integers(0, 8))
        gs = genes[int(rng.integers(len(genes)))]
        L = int(rng.integers(60, 220))
        p = int(rng.integers(0, max(1, len(gs) - 80)))
        piece = gs[p:p + L]
        if kind == 0:
            t = mutate(piece, int(rng.integers(0, 6)), 0)
        elif kind == 1:
            t = mutate(piece, int(rng.integers(0, 4)), int(rng.integers(1, 4)))
        elif kind == 2:     # V end + random junction + J start of one chain type: the short-anchor rescue (GetVJOverlapsFromHits)
            vn, v = vjs_v[int(rng.integers(len(vjs_v)))]
            cand = [x for x in vjs_j if x[0][:3] == vn[:3]] or vjs_j
            j = cand[int(rng.integers(len(cand)))][1]
            t = v[-int(rng.integers(18, 30)):] + rnd(int(rng.integers(3, 15))) + j[: int(rng.integers(18, 30))]
        elif kind == 3:
            t = "".join(comp[c] for c in reversed(mutate(piece, 2, int(rng.integers(0, 2)))))
        elif kind == 4:
            t = rnd(L)
        elif kind == 5:
            g2 = genes[int(rng.integers(len(genes)))]
            t = piece[: L // 2] + g2[-(L // 2):]
        elif kind == 6:     # a long unmatched stretch between two anchors of the same gene: gap alignment
            q = min(len(piece) - 30, 40)
            t = piece[:q] + mutate(piece[q:q + 40], 12, 0) + piece[q + 40:]
        else:
            t = piece
        reads.append(t[:400] if len(t) >= 1 else "A")
    n_ovl = n_reads = n_vj = n_indel = 0
    for i, t in enumerate(reads):
        gn, go, gsim = g.get_overlaps(t)
        rn, ro, rsim = r.get_overlaps(t, 0, -1, False)
        assert gn == rn, ("count", i, gn, rn, t)
        if rn > 0:
            assert (go == ro).all(), ("overlap", i, go, ro, t)
            assert (gsim == rsim).all(), ("similarity", i)
            n_ovl += rn
            n_reads += 1
            n_indel += int((go[:, 7] > 0).any())          # go equals ro
    assert n_reads > n // 3 and n_ovl > n and (n_indel > 5 or radius == 0), (n_reads, n_ovl, n_indel)
    g.close()
    return n_ovl


def check_refset_annotate(lib, ref, tmp_path, seed=141, n=600, radius=None, hit_len=31, k=9):
    """t4_refset_annotate against SeqSet::AnnotateRead(read, 0, geneOverlap, NULL, NULL) -- the rough annotation the stage-1
    driver runs on every read (main.cpp:1084-1120): per gene type V / D / J / C the chosen gene, coordinates, strand, matchCnt,
    indelCnt, similarity.  Reads: clonotype reads (V + junction + J + C in one read), mutated gene pieces, V/J-only ends,
    reverse strands, chimeras of two chains (one chain per read rule), random reads, reads cut into several contigs by runs
    of N's, short constant-gene matches."""
    rng = np.random.default_rng(seed)
    fa = os.path.join(str(tmp_path), "genes_a%d.fa" % seed)
    recs = write_gene_fasta(fa)
    lib.check(lib.reset())
    g = api.RefSet(fa, k, lib, hit_len_required=hit_len)
    r = ref.RefGeneSet(fa, k, hit_len_required=hit_len)
    if radius is not None:
        g.set_radius(radius)
        r.set_radius(radius)
    cl = synth.make_clones(60, seed)
    rd = synth.sample_pairs(cl, n // 3, 150, seed, sub_rate=0.02)
    reads = [synth.decode(c) for c in rd.codes]
    comp = {"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}
    genes = [s for _, s in recs if len(s) > 200]
    cgenes = [s for nm, s in recs if len(nm) > 3 and nm[3] not in "VDJ" and len(s) > 150]
    src = list(reads)

    def rnd(L):
        return "".join("ACGT"[c] for c in rng.integers(0, 4, size=L))

    while len(reads) < n:
        kind = int(rng.integers(0, 8))
        base = src[int(rng.integers(len(src)))]
        gs = genes[int(rng.integers(len(genes)))]
        p = int(rng.integers(0, max(1, len(gs) - 80)))
        piece = gs[p:p + int(rng.integers(60, 200))]
        if kind == 0:       # a run of N's splits the read into contigs
            q = int(rng.integers(20, len(base) - 30))
            t = base[:q] + "N" * int(rng.integers(7, 15)) + base[q + 10:]
        elif kind == 1:     # sparse N's: still one contig
            t = list(base)
            for q in rng.integers(0, len(t), size=int(rng.integers(1, 6))):
                t[int(q)] = "N"
            t = "".join(t)
        elif kind == 2:
            t = "".join(comp[c] for c in reversed(base))
        elif kind == 3:     # two chains in one read
            o = src[int(rng.integers(len(src)))]
            t = base[:75] + o[75:]
        elif kind == 4:
            t = rnd(int(rng.integers(40, 200)))
        elif kind == 5:     # V or J piece followed by a short constant-gene piece deep inside the gene
            c = cgenes[int(rng.integers(len(cgenes)))]
            q = int(rng.integers(100, max(101, len(c) - 45)))
            t = piece[:90] + c[q:q + int(rng.integers(30, 45))]
        elif kind == 6:
            t = piece
        else:
            t = base[: int(rng.integers(30, 100))]
        reads.append(t[:400])
    lens = np.array([len(x) for x in reads], dtype=np.int32)
    off = np.zeros(len(reads), dtype=np.uint64)
    off[1:] = np.cumsum(lens[:-1])
    pool = np.frombuffer(("".join(reads) + "\0" * 16).encode(), dtype=np.uint8).copy()
    go, gsim = g.annotate(pool, off, lens)
    n_set = np.zeros(4, dtype=np.int64)
    for i, t in enumerate(reads):
        ro, rsim = r.annotate_read(t)
        assert (go[i][:, 0] == ro[:, 0]).all(), ("gene", i, go[i][:, 0], ro[:, 0], t)
        for tt in range(4):
            if ro[tt, 0] >= 0:
                assert (go[i][tt] == ro[tt]).all() and gsim[i][tt] == rsim[tt], ("overlap", i, tt, go[i][tt], ro[tt], gsim[i][tt], rsim[tt], t)
                n_set[tt] += 1
            else:
                assert go[i][tt][5] == 1       # strand of an unset entry
    assert n_set[0] > n // 5 and n_set[2] > n // 20 and n_set[3] > n // 10, n_set
    g.close()
    return int(n_set.sum())


def check_sort_reads(lib, ref, seed=151, n=5000):
    """t4_sort_reads against std::sort with the driver's _sortRead::operator< (main.cpp:103-125, 1078): reads with their real
    k-mer statistics plus adversarial ties -- equal statistics with different strings, prefixes of each other, identical
    reads under different ids (mates, the '.1' copies), negative statistics, N's."""
    rng = np.random.default_rng(seed)
    cl = synth.make_clones(40, seed)
    rd = synth.sample_pairs(cl, n // 4, 150, seed, sub_rate=0.01)
    reads = [synth.decode(c) for c in rd.codes]
    ids = ["r%d" % (i // 2) for i in range(len(reads))]                 # mates share an id (main.cpp:1069)
    src = list(reads)
    while len(reads) < n:
        kind = int(rng.integers(0, 6))
        s = src[int(rng.integers(len(src)))]
        if kind == 0:
            t = s[: int(rng.integers(20, 150))]
        elif kind == 1:
            t = s
        elif kind == 2:
            t = list(s)
            t[int(rng.integers(len(t)))] = "N"
            t = "".join(t)
        elif kind == 3:
            t = "".join("ACGT"[c] for c in rng.integers(0, 4, size=int(rng.integers(10, 160))))
        elif kind == 4:
            t = s[:75]
        else:
            t = s[10:]
        reads.append(t)
        ids.append(("r%d" % int(rng.integers(0, n))) + (".1" if rng.random() < 0.2 else ""))
    lens = np.array([len(x) for x in reads], dtype=np.int32)
    off = np.zeros(len(reads), dtype=np.uint64)
    off[1:] = np.cumsum(lens[:-1])
    pool = np.frombuffer(("".join(reads) + "\0" * 16).encode(), dtype=np.uint8).copy()
    mn, med, avg, _ = ref.kmer_count_stats(pool, off, lens, 21)
    # coarsen a part of the statistics so that long runs of equal (min, median, avg, len) must be decided by the strings
    coarse = rng.random(len(reads)) < 0.5
    mn = np.where(coarse, np.minimum(mn, 2), mn).astype(np.int32)
    med = np.where(coarse, np.minimum(med, 3), med).astype(np.int32)
    avg = np.where(coarse, np.float32(2.5), avg).astype(np.float32)
    ro = ref.sort_reads(reads, ids, mn, med, avg)
    go = api.sort_reads(pool, off, lens, ids, mn, med, avg, lib)
    key = lambda i: (reads[i], ids[i], int(mn[i]), int(med[i]), float(avg[i]))
    assert sorted(go.tolist()) == list(range(len(reads)))
    # records that compare equal in every field may come in either order: compare the sorted RECORDS, not the indices
    assert [key(i) for i in go] == [key(i) for i in ro], np.flatnonzero(np.array([key(i) != key(j) for i, j in zip(go, ro)]))[:5]
    return len(reads)


def check_mate_overlap(lib, ref, seed=161, n=3000):
    """t4_mate_overlap_batch against AlignAlgo::IsMateOverlap (AlignAlgo.hpp:1027-1096): return value, offset, bestMatchCnt
    for overlapping mates (with mismatches), read-through pairs, unrelated pairs, tandem repeats, both checkTandem settings
    and the two minOverlap formulas of ProcessRead (main.cpp:244-249)."""
    rng = np.random.default_rng(seed)

    def rnd(L):
        return "".join("ACGT"[c] for c in rng.integers(0, 4, size=L))

    fr, sr = [], []
    for i in range(n):
        kind = int(rng.integers(0, 6))
        L1, L2 = int(rng.integers(30, 160)), int(rng.integers(30, 160))
        if kind == 0:       # suffix of f = prefix of s
            ov = int(rng.integers(5, min(L1, L2)))
            f = rnd(L1)
            s = f[L1 - ov:] + rnd(L2 - ov)
        elif kind == 1:     # the same with a few mismatches
            ov = int(rng.integers(10, min(L1, L2)))
            f = rnd(L1)
            t = list(f[L1 - ov:])
            for q in rng.integers(0, ov, size=int(rng.integers(1, 5))):
                t[int(q)] = "ACGT"[int(rng.integers(4))]
            s = "".join(t) + rnd(L2 - ov)
        elif kind == 2:     # read-through: s inside f
            f = rnd(L1)
            st = int(rng.integers(0, L1 // 2))
            s = f[st:st + L2]
        elif kind == 3:     # tandem repeats
            u = rnd(int(rng.integers(1, 5)))
            f = rnd(L1 // 2) + u * 20
            s = u * 20 + rnd(L2 // 2)
        elif kind == 4:
            f, s = rnd(L1), rnd(L2)
        else:               # two candidate offsets: ambiguous
            core = rnd(25)
            f = rnd(20) + core + rnd(15) + core
            s = core + rnd(L2)
        fr.append(f)
        sr.append(s)
    reads = fr + sr
    lens = np.array([len(x) for x in reads], dtype=np.int32)
    off = np.zeros(len(reads), dtype=np.uint64)
    off[1:] = np.cumsum(lens[:-1])
    pool = np.frombuffer(("".join(reads) + "\0" * 16).encode(), dtype=np.uint8).copy()
    fo, so = off[:n].copy(), off[n:].copy()
    fl, sl = lens[:n].copy(), lens[n:].copy()
    tot = fl + sl
    mo = np.where(rng.random(n) < 0.5, np.minimum(tot // 10, 31), np.minimum(tot // 20, 31)).astype(np.int32)
    ct = (rng.random(n) < 0.6).astype(np.uint8)
    gos, gof, gbm = (np.zeros(n, dtype=np.int32) for _ in range(3))
    lib.check(lib.mate_overlap_batch(pool.ctypes.data, pool.nbytes, fo.ctypes.data, fl.ctypes.data, so.ctypes.data, sl.ctypes.data, mo.ctypes.data,
                                     ct.ctypes.data, n, gos.ctypes.data, gof.ctypes.data, gbm.ctypes.data))
    n_pos = 0
    for i in range(n):
        r, o, b = ref.is_mate_overlap(fr[i], sr[i], int(mo[i]), int(ct[i]))
        assert (r, o, b) == (int(gos[i]), int(gof[i]), int(gbm[i])), (i, r, o, b, gos[i], gof[i], gbm[i], fr[i], sr[i])
        n_pos += r >= 0
    assert n_pos > n // 5 and n_pos < n
    return n_pos
