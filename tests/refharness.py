"""ctypes binding of the library-level oracle oracle/_ref/libt4ref.so (TEST INFRASTRUCTURE).

The oracle is compiled from the reference's sources, which are not part of this repository.  So that the parity tests
still compare against the reference where it cannot be built, every call of this module goes through a tape:

  live    oracle/_ref/libt4ref.so present: the reference computes every result;
  record  live, and T4_REF_RECORD=<dir> set: the results are also written to <dir>/<test>.xz;
  replay  no oracle: the results come from tests/golden/ref/<test>.xz, recorded from the reference itself.

Every recorded call carries a digest of its inputs; a replayed call whose inputs differ from the recorded ones fails
(the recording is then stale: regenerate it where the reference sources exist, tests/golden/make_ref_tapes.sh).
Results the tests only compare for equality (Output texts, hit lists, overlaps, LIS) are recorded as digests (OutputDigest,
ArrayDigest), which compare equal to what they were made from."""
import ctypes as C
import hashlib
import json
import lzma
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "libt4ref.so")
TAPES = os.path.join(ROOT, "tests", "golden", "ref")


def available():
    return os.path.exists(LIB)


def tape_path(test_id, directory=TAPES):
    """tests/golden/ref/<module>.<test>[-<params>].xz for a pytest node id."""
    mod, _, name = test_id.partition("::")
    name = re.sub(r"[^A-Za-z0-9_.]+", "-", name).strip("-")
    return os.path.join(directory, os.path.splitext(os.path.basename(mod))[0] + "." + name + ".xz")


class OutputDigest:
    """A recorded Output text: equal to the bytes whose SHA-256 it holds, and as long as they were."""
    __array_ufunc__ = None
    __hash__ = None

    def __init__(self, sha, n):
        self.sha, self.n = sha, n

    def __len__(self):
        return self.n

    def __eq__(self, other):
        if isinstance(other, OutputDigest):
            return (self.sha, self.n) == (other.sha, other.n)
        if isinstance(other, (bytes, bytearray)):
            return len(other) == self.n and _sha(other) == self.sha
        return NotImplemented

    def __ne__(self, other):
        eq = self.__eq__(other)
        return eq if eq is NotImplemented else not eq

    def __repr__(self):
        return "OutputDigest(%d bytes, sha256 %s)" % (self.n, self.sha[:16])


def canon_hits(h):
    """The reference's SortHits (SeqSet.hpp:1306) orders hits by (strand, seqIdx, readOffset) and leaves hits of
    one k-mer on one contig in postings (insertion) order, which nothing downstream observes
    (GetOverlapsFromHits re-sorts every group by diagonal).  Compare in the canonical order
    (strand, seqIdx, readOffset, seqOffset) the C ABI documents."""
    if isinstance(h, HitsDigest):
        return h.canon5
    if len(h) == 0:
        return h
    order = np.lexsort((h[:, 1], h[:, 2], h[:, 0], h[:, 3]))
    return h[order]


def canon4(h):
    """The first four columns of a hit list (no postings count), in the canonical order."""
    if isinstance(h, HitsDigest):
        return h.canon4
    if len(h) == 0:
        return h[:, :4]
    h = h[:, :4]
    return h[np.lexsort((h[:, 1], h[:, 2], h[:, 0], h[:, 3]))]


# results the tests only count and compare for equality: recorded as SHA-256 digests (hit lists in their canonical forms)
DIGESTED = ("get_overlaps", "lis")


def _sha(x):
    """64 bits of SHA-256: enough to tell a recorded result from a different one."""
    return hashlib.sha256(x if isinstance(x, (bytes, bytearray)) else np.ascontiguousarray(x).tobytes()).hexdigest()[:16]


class ArrayDigest:
    """A recorded array: its shape, and equal (a numpy bool) to the arrays of its dtype and SHA-256."""
    __array_ufunc__ = None
    __hash__ = None

    def __init__(self, sha, dtype, shape):
        self.sha, self.dtype, self.shape = sha, np.dtype(dtype), tuple(shape)

    def __len__(self):
        return self.shape[0]

    def __eq__(self, other):
        other = np.asarray(other)
        return np.bool_(other.shape == self.shape and _sha(other.astype(self.dtype, copy=False)) == self.sha)

    def __repr__(self):
        return "ArrayDigest(%s%s, sha256 %s)" % (self.dtype, self.shape, self.sha[:16])


class HitsDigest:
    """A recorded hit list: what canon_hits and canon4 give for it, as ArrayDigests."""

    def __init__(self, sha5, sha4, n):
        self.canon5, self.canon4 = ArrayDigest(sha5, "<i4", (n, 5)), ArrayDigest(sha4, "<i4", (n, 4))


class _File(str):
    """A path argument: the digest covers the file's content, not its (temporary) name."""


def _digest(h, x):
    if isinstance(x, _File):
        h.update(b"F" + open(x, "rb").read())
    elif isinstance(x, RefSeqSet):
        h.update(b"S%d" % x.id)
    elif isinstance(x, np.ndarray) and x.dtype.names:       # record arrays: the fields, not the bytes that pad them
        h.update(b"R")
        for n in x.dtype.names:
            _digest(h, x[n])
    elif isinstance(x, np.ndarray):
        x = np.ascontiguousarray(x)
        h.update(("A%s%s" % (x.dtype.str, x.shape)).encode() + x.tobytes())
    elif isinstance(x, (bytes, bytearray)):
        h.update(b"B%d:" % len(x) + bytes(x))
    elif isinstance(x, (list, tuple)):
        h.update(b"L%d" % len(x))
        for y in x:
            _digest(h, y)
    else:
        h.update(("V" + repr(x.item() if isinstance(x, np.generic) else x)).encode())


class Tape:
    """The sequence of oracle calls of one test: recorded live, or replayed from tests/golden/ref."""

    def __init__(self, path, record):
        self.path, self.record, self.entries, self.blob, self.nblob, self.pos = path, record, [], [], 0, 0
        if not record and os.path.exists(path):
            data = lzma.decompress(open(path, "rb").read())
            n = data.index(b"\n")
            self.entries, self.blob = json.loads(data[:n]), data[n + 1:]

    def call(self, name, args, fn):
        h = hashlib.sha256()
        _digest(h, args)
        key = h.hexdigest()[:10]
        if self.record:
            out = fn()
            self.entries.append([name, key, self._enc(out, name)])
            return out
        if not os.path.exists(self.path):
            raise FileNotFoundError("no recorded oracle results %s (oracle/_ref/libt4ref.so not built)" % os.path.relpath(self.path, ROOT))
        assert self.pos < len(self.entries), "oracle call %s beyond the recording %s" % (name, os.path.basename(self.path))
        rname, rkey, enc = self.entries[self.pos]
        assert (rname, rkey) == (name, key), ("oracle call %d of %s: %s with these inputs was not recorded (recorded: %s); "
                                              "the recording is stale" % (self.pos, os.path.basename(self.path), name, rname))
        self.pos += 1
        return self._dec(enc)

    def _enc(self, x, name=""):
        if name == "get_hits":
            return {"hits": [_sha(canon_hits(x)), _sha(canon4(x)), len(x)]}
        if name in DIGESTED and isinstance(x, np.ndarray):
            return {"digest": [_sha(x), x.dtype.str, list(x.shape)]}
        if x is None or isinstance(x, (bool, int, float, str)):
            return x
        if isinstance(x, np.generic):
            return {"n": x.dtype.str, "v": x.item()}
        if isinstance(x, (bytes, bytearray)):
            return {"h": _sha(x), "len": len(x)}
        if isinstance(x, np.ndarray):
            x = np.ascontiguousarray(x)
            self.blob.append(x.tobytes())
            self.nblob += x.nbytes
            return {"a": [x.dtype.str, list(x.shape), self.nblob - x.nbytes]}
        if isinstance(x, RefSeqSet):
            return {"set": x.id}
        if isinstance(x, tuple):
            return {"t": [self._enc(y, name) for y in x]}
        if isinstance(x, list):
            return {"l": [self._enc(y) for y in x]}
        if isinstance(x, dict):
            return {"d": {k: self._enc(v) for k, v in x.items()}}
        raise TypeError("cannot record %r" % type(x))

    def _dec(self, x):
        if not isinstance(x, dict):
            return x
        if "n" in x:
            return np.dtype(x["n"]).type(x["v"])
        if "h" in x:
            return OutputDigest(x["h"], x["len"])
        if "a" in x:
            dt, shape, o = x["a"]
            return np.frombuffer(self.blob, dtype=dt, count=int(np.prod(shape)), offset=o).reshape(shape).copy()
        if "hits" in x:
            return HitsDigest(*x["hits"])
        if "digest" in x:
            return ArrayDigest(*x["digest"])
        if "set" in x:
            return RefSeqSet(handle=0)
        if "t" in x:
            return tuple(self._dec(y) for y in x["t"])
        if "l" in x:
            return [self._dec(y) for y in x["l"]]
        return {k: self._dec(v) for k, v in x["d"].items()}

    def save(self):
        os.makedirs(os.path.dirname(self.path), exist_ok=True)
        data = json.dumps(self.entries, separators=(",", ":")).encode() + b"\n" + b"".join(self.blob)
        open(self.path, "wb").write(lzma.compress(data, preset=9 | lzma.PRESET_EXTREME))


_tape = None
_next_id = [0]


def use_tape(test_id):
    """Start the oracle calls of one test (a pytest node id): live, record or replay as the module docstring says."""
    global _tape
    _next_id[0] = 0
    rec = os.environ.get("T4_REF_RECORD")
    if available():
        _tape = Tape(tape_path(test_id, rec), True) if rec else None
    else:
        _tape = Tape(tape_path(test_id), False)
    return _tape


def end_tape():
    """Close the tape of a test: save a recording; a replay must have used every recorded call."""
    global _tape
    t, _tape = _tape, None
    if t is not None and t.record and t.entries:
        t.save()
    if t is not None and not t.record:
        assert t.pos == len(t.entries), ("%s: only %d of the %d recorded oracle calls were made; the recording is stale"
                                         % (os.path.basename(t.path), t.pos, len(t.entries)))


if __name__ == "__main__":
    # python tests/refharness.py tests/golden/ref/<tape>.xz: list the recorded calls (name, input digest, result)
    import sys
    t = Tape(sys.argv[1], False)
    for i, (name, key, enc) in enumerate(t.entries):
        r = repr(t._dec(enc))
        print("%5d %-26s %s  %s" % (i, name, key, r if len(r) < 200 else r[:200] + " ..."))


def _call(name, args, fn):
    if _tape is None:
        return fn()
    return _tape.call(name, args, fn)


_lib = None


def lib():
    global _lib
    if _lib is None:
        l = C.CDLL(LIB)
        l.t4ref_create.restype = C.c_void_p
        l.t4ref_create.argtypes = [C.c_int]
        l.t4ref_destroy.argtypes = [C.c_void_p]
        l.t4ref_set_hit_len_required.argtypes = [C.c_void_p, C.c_int]
        l.t4ref_set_novel_seq_similarity.argtypes = [C.c_void_p, C.c_double]
        l.t4ref_set_novel_seq_similarity.restype = C.c_double
        l.t4ref_size.argtypes = [C.c_void_p]
        l.t4ref_merge_sets.restype = C.c_void_p
        l.t4ref_merge_sets.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.POINTER(C.c_int)]
        l.t4ref_input_contig.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_void_p, C.c_int, C.c_int]
        l.t4ref_set_consider_barcode_in_hash.argtypes = [C.c_void_p, C.c_int]
        l.t4ref_reverse_complement_in_place.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        l.t4ref_kmer_length.argtypes = [C.c_void_p]
        l.t4ref_add_read.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.c_double]
        l.t4ref_repeat_add_read.argtypes = [C.c_void_p, C.c_char_p]
        l.t4ref_input_novel_read.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int, C.c_int]
        l.t4ref_update_all_consensus.argtypes = [C.c_void_p]
        l.t4ref_change_kmer_length.argtypes = [C.c_void_p, C.c_int]
        l.t4ref_has_motif.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        l.t4ref_output_mem.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        l.t4ref_free.argtypes = [C.c_void_p]
        l.t4ref_get_hits.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
        l.t4ref_get_chains.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                       C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        l.t4ref_get_overlaps.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        l.t4ref_dp_pos_weight.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.c_void_p]
        l.t4ref_index_lookup.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_int]
        l.t4ref_index_checksum.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        l.t4ref_index_checksum.restype = C.c_int64
        l.t4ref_nomatch_gap_limit.argtypes = [C.c_void_p]
        l.t4ref_get_contig.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.c_void_p, C.c_char_p, C.c_int,
                                       C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
        l.t4ref_run_descs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_char_p), C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_void_p]
        l.t4ref_release_finished_barcode.argtypes = [C.c_void_p, C.c_int, C.c_int]
        l.t4ref_release_shallow_contigs.argtypes = [C.c_void_p, C.c_int]
        l.t4ref_input_novel_fa.argtypes = [C.c_void_p, C.c_char_p]
        l.t4ref_num_read.argtypes = [C.c_void_p, C.c_int]
        l.t4ref_kmer_count_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p]
        l.t4ref_refset_create.restype = C.c_void_p
        l.t4ref_refset_create.argtypes = [C.c_char_p, C.c_int]
        l.t4ref_seq_name.restype = C.c_char_p
        l.t4ref_seq_name.argtypes = [C.c_void_p, C.c_int]
        l.t4ref_seq_count.argtypes = [C.c_void_p]
        l.t4ref_set_radius.argtypes = [C.c_void_p, C.c_int]
        l.t4ref_has_hit_in_set.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        l.t4ref_is_low_complexity.argtypes = [C.c_char_p]
        l.t4ref_annotate_read.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p]
        l.t4ref_sort_reads.argtypes = [C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        l.t4ref_is_mate_overlap.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        l.t4ref_lis.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        l.t4ref_input_seqset.restype = C.c_void_p
        l.t4ref_input_seqset.argtypes = [C.c_void_p, C.c_int]
        l.t4ref_assign_read.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_double)]
        l.t4ref_assign_pass.restype = C.c_void_p
        l.t4ref_assign_pass.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                        C.c_void_p, C.c_void_p]
        _lib = l
    return _lib


class RefSeqSet:
    """The reference SeqSet (compiled from the reference sources) behind the same call names as trust4_b200.api.SeqSet."""

    def __init__(self, k=9, handle=None):
        self.id = _next_id[0]
        _next_id[0] += 1
        self.l = lib() if available() else None
        self.h = handle if handle is not None else (self.l.t4ref_create(k) if self.l else 0)

    def close(self):
        if self.h:
            self.l.t4ref_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def _call(self, name, args, fn):
        return _call(name, (self,) + tuple(args), fn)

    def set_hit_len_required(self, v):
        return self._call("set_hit_len_required", (v,), lambda: self.l.t4ref_set_hit_len_required(self.h, v))

    def set_consider_barcode_in_hash(self, v):
        return self._call("set_consider_barcode_in_hash", (v,), lambda: self.l.t4ref_set_consider_barcode_in_hash(self.h, v))

    def size(self):
        return self._call("size", (), lambda: self.l.t4ref_size(self.h))

    def kmer_length(self):
        return self._call("kmer_length", (), lambda: self.l.t4ref_kmer_length(self.h))

    def add_read(self, read, name, strand, barcode, min_kmer_count, repetitive, thr):
        def f():
            s = C.c_int(strand)
            r = self.l.t4ref_add_read(self.h, read.encode(), name.encode(), C.byref(s), barcode, min_kmer_count, int(repetitive), thr)
            return r, s.value
        return self._call("add_read", (read, name, strand, barcode, min_kmer_count, repetitive, thr), f)

    def repeat_add_read(self, read):
        return self._call("repeat_add_read", (read,), lambda: self.l.t4ref_repeat_add_read(self.h, read.encode()))

    def input_novel_read(self, name, read, strand, barcode):
        return self._call("input_novel_read", (name, read, strand, barcode),
                          lambda: self.l.t4ref_input_novel_read(self.h, name.encode(), read.encode(), strand, barcode))

    def update_all_consensus(self):
        self._call("update_all_consensus", (), lambda: self.l.t4ref_update_all_consensus(self.h))

    def change_kmer_length(self, k):
        self._call("change_kmer_length", (k,), lambda: self.l.t4ref_change_kmer_length(self.h, k))

    def release_finished_barcode(self, barcode, contig_min_cov=0):
        self._call("release_finished_barcode", (barcode, contig_min_cov),
                   lambda: self.l.t4ref_release_finished_barcode(self.h, barcode, contig_min_cov))

    def release_shallow_contigs(self, min_cov):
        self._call("release_shallow_contigs", (min_cov,), lambda: self.l.t4ref_release_shallow_contigs(self.h, min_cov))

    def input_novel_fa(self, filename):
        self._call("input_novel_fa", (_File(filename),), lambda: self.l.t4ref_input_novel_fa(self.h, filename.encode()))

    def num_read(self, slot):
        return self._call("num_read", (slot,), lambda: self.l.t4ref_num_read(self.h, slot))

    def has_motif(self, read, strand):
        return self._call("has_motif", (read, strand), lambda: self.l.t4ref_has_motif(self.h, read.encode(), strand))

    def output(self):
        def f():
            buf = C.c_void_p()
            n = C.c_size_t()
            self.l.t4ref_output_mem(self.h, C.byref(buf), C.byref(n))
            s = C.string_at(buf, n.value)
            self.l.t4ref_free(buf)
            return s
        return self._call("output", (), f)

    def get_hits(self, read, strand=0, barcode=-1, allow_total_skip=False, cap=1 << 20):
        def f():
            out = np.zeros((cap, 5), dtype=np.int32)
            n = self.l.t4ref_get_hits(self.h, read.encode(), strand, barcode, int(allow_total_skip), out.ctypes.data, cap)
            assert n <= cap
            return out[:n].copy()
        return self._call("get_hits", (read, strand, barcode, allow_total_skip), f)

    def get_chains(self, read, strand=0, barcode=-1, allow_total_skip=False, filt=1, cap=1 << 14, ccap=1 << 20):
        def f():
            out = np.zeros((cap, 8), dtype=np.int32)
            co = np.zeros((ccap, 2), dtype=np.int32)
            nc = C.c_int()
            n = self.l.t4ref_get_chains(self.h, read.encode(), strand, barcode, int(allow_total_skip), filt, out.ctypes.data, cap,
                                        co.ctypes.data, ccap, C.byref(nc))
            assert n <= cap and nc.value <= ccap
            return out[:n].copy(), co[:nc.value].copy()
        return self._call("get_chains", (read, strand, barcode, allow_total_skip, filt), f)

    def get_overlaps(self, read, strand=0, barcode=-1, skip_repeats=False, cap=1 << 14):
        def f():
            out = np.zeros((cap, 8), dtype=np.int32)
            sim = np.zeros(cap, dtype=np.float64)
            n = self.l.t4ref_get_overlaps(self.h, read.encode(), strand, barcode, int(skip_repeats), out.ctypes.data, sim.ctypes.data, cap)
            if n < 0:
                return n, None, None
            return n, out[:n].copy(), sim[:n].copy()
        return self._call("get_overlaps", (read, strand, barcode, skip_repeats), f)

    def index_lookup(self, code, barcode=-1, cap=1 << 20):
        def f():
            out = np.zeros((cap, 2), dtype=np.int32)
            n = self.l.t4ref_index_lookup(self.h, code, barcode, out.ctypes.data, cap)
            return out[:n].copy()
        return self._call("index_lookup", (code, barcode), f)

    def index_checksum(self):
        def f():
            cs = C.c_uint64()
            n = self.l.t4ref_index_checksum(self.h, C.byref(cs))
            return n, cs.value
        return self._call("index_checksum", (), f)

    def get_contig(self, slot):
        def f():
            ln = self.l.t4ref_get_contig(self.h, slot, None, 0, None, None, 0, None, None, None, None)
            if ln < 0:
                return None
            cons = C.create_string_buffer(ln + 1)
            pw = np.zeros((ln, 4), dtype=np.int32)
            name = C.create_string_buffer(4096)
            bc, nr, ml, mr = C.c_int(), C.c_int(), C.c_int(), C.c_int()
            self.l.t4ref_get_contig(self.h, slot, cons, ln + 1, pw.ctypes.data, name, 4096, C.byref(bc), C.byref(nr), C.byref(ml), C.byref(mr))
            return dict(consensus=cons.value.decode(), pos_weight=pw, name=name.value.decode(), barcode=bc.value,
                        num_read=nr.value, min_left=ml.value, min_right=mr.value)
        return self._call("get_contig", (slot,), f)

    def run_descs(self, cfg, descs, pool, names):
        descs = np.ascontiguousarray(descs)
        pool = np.ascontiguousarray(pool)

        def f():
            n = len(descs)
            ret = np.zeros(n, dtype=np.int32)
            strands = np.zeros(n, dtype=np.int8)
            resc = np.zeros(n, dtype=np.int32)
            arr = (C.c_char_p * max(1, len(names)))(*names)
            a = self.l.t4ref_run_descs(self.h, cfg.ctypes.data, descs.ctypes.data, n, pool.ctypes.data, arr, len(names),
                                       ret.ctypes.data, strands.ctypes.data, resc.ctypes.data)
            return a, ret, strands, resc
        return self._call("run_descs", (cfg, descs, pool, list(names)), f)


def dp_pos_weight(tw, p):
    """AlignAlgo::GlobalAlignment_PosWeight via the reference; returns (score, edit list)."""
    tw = np.ascontiguousarray(tw, dtype=np.int32)

    def f():
        lent, lenp = tw.shape[0], len(p)
        al = np.zeros(lent + lenp + 4, dtype=np.int8)
        sc = lib().t4ref_dp_pos_weight(tw.ctypes.data, lent, p.encode(), lenp, al.ctypes.data)
        e = []
        for v in al:
            if v == -1:
                break
            e.append(int(v))
        return sc, e
    return _call("dp_pos_weight", (tw, p), f)


class RefGeneSet(RefSeqSet):
    """The reference's `SeqSet refSet(k); refSet.InputRefFa(fasta)` (fastq-extractor / trust4 reference gene set)."""

    def __init__(self, fasta, k=9, hit_len_required=27):
        super().__init__(k, handle=lib().t4ref_refset_create(fasta.encode(), k) if available() else 0)
        self._call("refset_create", (_File(fasta), k), lambda: None)
        self.set_hit_len_required(hit_len_required)

    def names(self):
        return self._call("names", (), lambda: [self.l.t4ref_seq_name(self.h, i).decode() for i in range(self.l.t4ref_seq_count(self.h))])

    def set_radius(self, r):
        self._call("set_radius", (r,), lambda: self.l.t4ref_set_radius(self.h, r))

    def annotate_read(self, read):
        """AnnotateRead(read, 0, ...): (int32[4, 8] for V, D, J, C; similarity[4])."""
        def f():
            out = np.zeros((4, 8), dtype=np.int32)
            sim = np.zeros(4, dtype=np.float64)
            self.l.t4ref_annotate_read(self.h, read.encode(), out.ctypes.data, sim.ctypes.data)
            return out, sim
        return self._call("annotate_read", (read,), f)

    def has_hit_in_set(self, read, mode=0):
        return self._call("has_hit_in_set", (read, mode), lambda: self.l.t4ref_has_hit_in_set(self.h, read.encode(), mode))


def is_low_complexity(read):
    return _call("is_low_complexity", (read,), lambda: lib().t4ref_is_low_complexity(read.encode()))


_helper = []


def _helper_set():
    """One reference SeqSet for the member functions that do not depend on the set's contents."""
    if not _helper:
        _helper.append(lib().t4ref_create(9))
    return _helper[0]


def reverse_complement(s):
    """SeqSet's reverse complement of the string s."""
    def f():
        b = C.create_string_buffer(s.encode())
        lib().t4ref_reverse_complement_in_place(_helper_set(), b, len(s))
        return b.value.decode()
    return _call("reverse_complement", (s,), f)


def lis(a, b):
    """SeqSet::LongestIncreasingSubsequence over the (a, b) pairs: the chosen pairs as two int32 arrays."""
    a = np.ascontiguousarray(a, dtype=np.int32)
    b = np.ascontiguousarray(b, dtype=np.int32)

    def f():
        ra, rb = np.zeros(len(a), dtype=np.int32), np.zeros(len(a), dtype=np.int32)
        n = lib().t4ref_lis(_helper_set(), a.ctypes.data, b.ctypes.data, len(a), ra.ctypes.data, rb.ctypes.data)
        return ra[:n].copy(), rb[:n].copy()
    return _call("lis", (a, b), f)


def is_mate_overlap(f_read, s_read, min_overlap, check_tandem):
    """AlignAlgo::IsMateOverlap: (return value, offset, bestMatchCnt)."""
    def f():
        o, b = C.c_int32(), C.c_int32()
        r = lib().t4ref_is_mate_overlap(f_read.encode(), len(f_read), s_read.encode(), len(s_read), min_overlap, check_tandem, C.byref(o), C.byref(b))
        return r, o.value, b.value
    return _call("is_mate_overlap", (f_read, s_read, min_overlap, check_tandem), f)


def kmer_count_stats(pool, seq_off, lens, k=21, qual=None):
    """The reference's KmerCount over the reads: (min, median, avg, new length) per read (KmerCount.hpp:64-97, 177-288)."""
    pool = np.ascontiguousarray(pool)
    seq_off = np.ascontiguousarray(seq_off, dtype=np.uint64)
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    if qual is not None:
        qual = np.ascontiguousarray(qual)

    def f():
        n = len(lens)
        mn = np.zeros(max(1, n), dtype=np.int32)
        med = np.zeros(max(1, n), dtype=np.int32)
        avg = np.zeros(max(1, n), dtype=np.float32)
        nl = np.zeros(max(1, n), dtype=np.int32)
        lib().t4ref_kmer_count_stats(pool.ctypes.data, qual.ctypes.data if qual is not None else None, seq_off.ctypes.data, lens.ctypes.data, n, k,
                                     mn.ctypes.data, med.ctypes.data, avg.ctypes.data, nl.ctypes.data)
        return mn[:n].copy(), med[:n].copy(), avg[:n].copy(), nl[:n].copy()
    return _call("kmer_count_stats", (pool, seq_off, lens, k, qual), f)


def sort_reads(reads, ids, min_cnt, median_cnt, avg_cnt):
    """std::sort with _sortRead::operator< (main.cpp:103-125): the permutation (order[j] = original index)."""
    min_cnt = np.ascontiguousarray(min_cnt, dtype=np.int32)
    median_cnt = np.ascontiguousarray(median_cnt, dtype=np.int32)
    avg_cnt = np.ascontiguousarray(avg_cnt, dtype=np.float32)

    def f():
        n = len(reads)
        ra = (C.c_char_p * max(1, n))(*[r.encode() for r in reads])
        ia = (C.c_char_p * max(1, n))(*[i.encode() for i in ids])
        order = np.zeros(max(1, n), dtype=np.int64)
        lib().t4ref_sort_reads(ra, ia, min_cnt.ctypes.data, median_cnt.ctypes.data, avg_cnt.ctypes.data, n, order.ctypes.data)
        return order[:n].copy()
    return _call("sort_reads", (list(reads), list(ids), min_cnt, median_cnt, avg_cnt), f)


def assembled_list(ret, resc):
    """The driver's assembledReadIdx (main.cpp:1779, 1933): reads added in the main pass, in order, then the rescued ones."""
    ret = np.asarray(ret)
    main = np.nonzero(ret >= 0)[0]
    if resc is None:
        return main.astype(np.int32)
    resc = np.asarray(resc)
    rescued = np.nonzero((resc != np.iinfo(np.int32).min) & (resc >= 0))[0]
    return np.concatenate([main, rescued]).astype(np.int32)


def assign_pass(src, k, descs, pool, lst, strands, recompute=True):
    """main.cpp:2047-2118 on the reference SeqSet `src`: (extended RefSeqSet, assign int32[n, 8], similarity[n]) per list element."""
    descs = np.ascontiguousarray(descs)
    pool = np.ascontiguousarray(pool)
    lst = np.ascontiguousarray(lst, dtype=np.int32)
    strands = np.ascontiguousarray(strands, dtype=np.int8)

    def f():
        n = len(lst)
        a = np.zeros((max(1, n), 8), dtype=np.int32)
        s = np.zeros(max(1, n), dtype=np.float64)
        h = lib().t4ref_assign_pass(src.h, k, descs.ctypes.data, pool.ctypes.data, lst.ctypes.data, n, strands.ctypes.data,
                                    int(recompute), a.ctypes.data, s.ctypes.data)
        return RefSeqSet(k, handle=h), a[:n].copy(), s[:n].copy()
    return _call("assign_pass", (src, k, descs, pool, lst, strands, recompute), f)


def merge_sets(shards, k=9):
    """SURVEY.md 8e(2) merge oracle over reference SeqSets in (rank, stream) order -> (merged RefSeqSet, n removed)."""
    def f():
        arr = (C.c_void_p * len(shards))(*[s.h for s in shards])
        removed = C.c_int()
        h = lib().t4ref_merge_sets(arr, len(shards), k, C.byref(removed))
        return RefSeqSet(k, handle=h), removed.value
    return _call("merge_sets", (list(shards), k), f)


def set_from_contigs(contigs, k=9):
    """Reference SeqSet holding the given contigs (dicts as produced by trust4_b200.dist.unpack_contigs)."""
    s = RefSeqSet(k)
    for c in contigs:
        pw = np.ascontiguousarray(c["pos_weight"], dtype=np.int32)
        _call("input_contig", (s, c["name"], c["consensus"], pw, c["barcode"], c["num_read"]),
              lambda: lib().t4ref_input_contig(s.h, c["name"].encode(), c["consensus"].encode(), pw.ctypes.data, c["barcode"], c["num_read"]))
    return s
