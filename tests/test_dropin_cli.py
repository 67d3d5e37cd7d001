"""The drop-in stage-1 binary: the UNMODIFIED reference main.cpp + integration/t4_seqset_adapter.hpp + this
repository's C-ABI library must write the same _raw.out, _final.out and _assembled_reads.fa as the stock `trust4`
(oracle/_ref/trust4) -- flags, file formats and `run-trust4 --stage 1` compatibility included (SURVEY.md 8b).

CPU variant: integration/_build/trust4_emu{,_batch}, the binding linked against the test emulation of the engine.
GPU variant: integration/_build/trust4_gpu{,_batch}, linked against libtrust4_b200.so.
All of them, and the stock binary, are compiled from the reference's main.cpp, which is not part of this repository:
__graft_entry__.build() builds them where the reference sources exist, and the tests use them wherever they were built.
Inputs are synthetic FASTQ generated here, or the reference's shipped example (tests/golden/*.gz)."""
import gzip
import os
import shutil
import subprocess

import pytest

from trust4_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STOCK = os.path.join(ROOT, "oracle", "_ref", "trust4")
GOLD = os.path.join(ROOT, "tests", "golden")
SUFFIXES = ("_raw.out", "_final.out", "_assembled_reads.fa")


def write_inputs(tmp, npairs=1500, nclones=40, seed=21):
    pool = synth.load_gene_pool()
    fa = os.path.join(tmp, "genes.fa")
    with open(fa, "w") as f:
        for ch in pool.values():
            for seg in ch.values():
                for name, seq in seg:
                    f.write(">%s\n%s\n" % (name, seq))
    cl = synth.make_clones(nclones, seed)
    rd = synth.sample_pairs(cl, npairs, 150, seed)
    synth.write_fastq(rd, os.path.join(tmp, "reads"))
    return ["-f", fa, "-1", os.path.join(tmp, "reads_1.fq"), "-2", os.path.join(tmp, "reads_2.fq")]


def write_barcode_inputs(tmp, nreads=1500, nclones=24, n_barcodes=6, seed=23):
    """10x-style single-end input (BASELINE configs[3] flavour): every read carries a cell barcode (--barcode file with
    the same ids); a cell = a few clonotypes, plus a few ambient reads of other cells' clones."""
    import numpy as np
    pool = synth.load_gene_pool()
    fa = os.path.join(tmp, "genes.fa")
    with open(fa, "w") as f:
        for ch in pool.values():
            for seg in ch.values():
                for name, seq in seg:
                    f.write(">%s\n%s\n" % (name, seq))
    cl = synth.make_clones(nclones, seed)
    rd = synth.sample_pairs(cl, nreads, 150, seed, paired=False)
    rng = np.random.default_rng(seed)
    bc = rd.clone % n_barcodes
    amb = rng.random(nreads) < 0.02
    bc = np.where(amb, rng.integers(0, n_barcodes, size=nreads), bc)
    tags = ["".join("ACGT"[c] for c in rng.integers(0, 4, size=16)) for _ in range(n_barcodes)]
    with open(os.path.join(tmp, "reads.fq"), "w") as fq, open(os.path.join(tmp, "bc.fa"), "w") as fb:
        for i in range(nreads):
            fq.write("@r%d\n%s\n+\n%s\n" % (i, synth.decode(rd.codes[i]), "I" * 150))
            fb.write(">r%d\n%s\n" % (i, tags[int(bc[i])]))
    return ["-f", fa, "-u", os.path.join(tmp, "reads.fq"), "--barcode", os.path.join(tmp, "bc.fa")]


def example_inputs(tmp):
    """BASELINE.json configs[0]: the reference's shipped example, example_1.fq + example_2.fq -f hg38_bcrtcr.fa."""
    paths = []
    for name in ("hg38_bcrtcr.fa", "example_1.fq", "example_2.fq"):
        paths.append(os.path.join(tmp, name))
        with gzip.open(os.path.join(GOLD, name + ".gz")) as src, open(paths[-1], "wb") as dst:
            shutil.copyfileobj(src, dst)
    return ["-f", paths[0], "-1", paths[1], "-2", paths[2]]


def run_and_compare(binary, args, tmp, extra=(), env=None):
    for exe, tag in ((STOCK, "stock"), (binary, "dropin")):
        e = dict(os.environ, **env) if (env and exe is binary) else None
        subprocess.run([exe, "-t", "1", "-o", os.path.join(tmp, tag)] + list(extra) + args, check=True,
                       stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=900, env=e)
    for suf in SUFFIXES:
        a = open(os.path.join(tmp, "stock" + suf), "rb").read()
        b = open(os.path.join(tmp, "dropin" + suf), "rb").read()
        assert len(a) > 0 and a == b, suf


def prebuilt(name):
    """integration/_build/<name> and the stock binary, as __graft_entry__.build() left them (both need the reference sources)."""
    binary = os.path.join(ROOT, "integration", "_build", name)
    if not (os.path.exists(binary) and os.path.exists(STOCK)):
        pytest.skip("drop-in / stock binaries not built: they are compiled from the reference's main.cpp")
    return binary


@pytest.fixture(scope="module")
def emu_binary(emu_lib):
    return prebuilt("trust4_emu")


@pytest.fixture(scope="module")
def emu_batch_binary(emu_lib):
    """The batch route: main.cpp + one inserted line per offloaded pass (integration/make_batch_main.py), T4_STREAMS selects the device streams."""
    return prebuilt("trust4_emu_batch")


def test_batch_emu_shipped_example(emu_batch_binary, tmp_path):
    """BASELINE.json configs[0] through the batch route, one stream: the device runs the whole loop + rescue pass in one
    launch, the driver's own loop replays its decisions; all three output files byte-identical to the stock binary."""
    run_and_compare(emu_batch_binary, example_inputs(str(tmp_path)), str(tmp_path), env={"T4_STREAMS": "1"})


def test_batch_emu_synthetic(emu_batch_binary, tmp_path):
    run_and_compare(emu_batch_binary, write_inputs(str(tmp_path)), str(tmp_path), env={"T4_STREAMS": "1"})


def test_batch_emu_assign_pass_on_device(emu_batch_binary, tmp_path):
    """The second offloaded pass of the batch route (SURVEY.md 8f-2): with paired-end bulk input the driver's AssignRead
    loop (main.cpp:2075-2116) is replaced by t4_streams_assign_reads; _final.out -- which the reference derives from those
    assignments through RecomputePosWeight and the mate extension -- must stay byte-identical, with the pass on the device
    (default) and with T4_ASSIGN=0 (the driver's own CPU loop)."""
    tmp = str(tmp_path)
    args = write_inputs(tmp, 2500, 80, 31)
    subprocess.run([STOCK, "-t", "1", "-o", os.path.join(tmp, "stock")] + args, check=True, stdout=subprocess.DEVNULL,
                   stderr=subprocess.DEVNULL, timeout=900)
    for tag, env in (("dev", {"T4_STREAMS": "1"}), ("cpu", {"T4_STREAMS": "1", "T4_ASSIGN": "0"})):
        r = subprocess.run([emu_batch_binary, "-t", "1", "-o", os.path.join(tmp, tag)] + args, check=True, stdout=subprocess.DEVNULL,
                           stderr=subprocess.PIPE, timeout=900, env=dict(os.environ, **env), text=True)
        assert ("AssignRead pass on the device" in r.stderr) == (tag == "dev")
        for suf in SUFFIXES:
            a = open(os.path.join(tmp, "stock" + suf), "rb").read()
            assert len(a) > 0 and a == open(os.path.join(tmp, tag + suf), "rb").read(), (tag, suf)


@pytest.mark.parametrize("case", ["synthetic", "example", "repseq"])
def test_batch_emu_annotate_on_device(emu_batch_binary, tmp_path, case):
    """The third pass of the batch route, opt-in with T4_ANNOTATE=1 (SURVEY.md 8f-1): the driver's rough annotation loop
    (main.cpp:1084-1120) is replaced by t4_refset_annotate on a gene set rebuilt on the device from the -f file.  With all
    three passes on the (emulated) device -- rough annotation, AddRead loop + rescue, AssignRead -- the three output files
    stay byte-identical to the stock binary's: synthetic pairs; the shipped example (BASELINE configs[0], hg38_bcrtcr.fa);
    --trimLevel 2 (gene set re-indexed at k = 7, radius 0, main.cpp:766-771, 1082-1083).  Emulation only: the device pass
    has not run on a GPU yet."""
    tmp = str(tmp_path)
    extra = []
    if case == "synthetic":
        args = write_inputs(tmp, 1500, 50, 33)
    elif case == "example":
        args = example_inputs(tmp)
    else:
        args = write_inputs(tmp, 800, 25, 34)
        extra = ["--trimLevel", "2", "--skipMateExtension"]
    subprocess.run([STOCK, "-t", "1", "-o", os.path.join(tmp, "stock")] + extra + args, check=True, stdout=subprocess.DEVNULL,
                   stderr=subprocess.DEVNULL, timeout=900)
    r = subprocess.run([emu_batch_binary, "-t", "1", "-o", os.path.join(tmp, "dev")] + extra + args, check=True, stdout=subprocess.DEVNULL,
                       stderr=subprocess.PIPE, timeout=900, env=dict(os.environ, T4_STREAMS="1", T4_ANNOTATE="1"), text=True)
    assert "rough annotation on the device" in r.stderr
    for suf in SUFFIXES:
        a = open(os.path.join(tmp, "stock" + suf), "rb").read()
        assert len(a) > 0 and a == open(os.path.join(tmp, "dev" + suf), "rb").read(), (case, suf)


def _degrade_qualities(prefix, seed=5):
    """Give a fifth of the reads of <prefix>_1.fq / _2.fq a low-quality tail (Phred 2) so that the quality trimming of
    GetCountStatsAndTrim (KmerCount.hpp:241-271, default --trimLevel 1) really cuts reads."""
    import numpy as np
    rng = np.random.default_rng(seed)
    for m in ("_1.fq", "_2.fq"):
        lines = open(prefix + m).read().split("\n")
        for i in range(3, len(lines), 4):
            if lines[i] and rng.random() < 0.2:
                q = int(rng.integers(len(lines[i]) // 2, len(lines[i])))
                lines[i] = lines[i][:q] + "#" * (len(lines[i]) - q)
                seq = list(lines[i - 2])             # bad bases are often wrong bases: the tail's k-mers become singletons
                for x in range(q, len(seq)):
                    if rng.random() < 0.3:
                        seq[x] = "ACGT"[int(rng.integers(4))]
                lines[i - 2] = "".join(seq)
        open(prefix + m, "w").write("\n".join(lines))


def test_batch_emu_all_passes_on_device(emu_batch_binary, tmp_path):
    """Every pass the batch route can offload, together (T4_KMERSTATS=1 T4_SORT=1 T4_ANNOTATE=1 on top of the defaults): 21-mer
    statistics with quality trimming (main.cpp:981-1010), the read sort (:1078), rough annotation (:1084-1120), AddRead loop +
    rescue (:1583-1940), AssignRead
    (:2075-2116) -- on reads whose tails really get trimmed.  The three output files equal the stock binary's byte for byte."""
    tmp = str(tmp_path)
    args = write_inputs(tmp, 1500, 50, 35)
    _degrade_qualities(os.path.join(tmp, "reads"))
    subprocess.run([STOCK, "-t", "1", "-o", os.path.join(tmp, "stock")] + args, check=True, stdout=subprocess.DEVNULL,
                   stderr=subprocess.DEVNULL, timeout=900)
    r = subprocess.run([emu_batch_binary, "-t", "1", "-o", os.path.join(tmp, "dev")] + args, check=True, stdout=subprocess.DEVNULL,
                       stderr=subprocess.PIPE, timeout=900, env=dict(os.environ, T4_STREAMS="1", T4_ANNOTATE="1", T4_KMERSTATS="1", T4_SORT="1"), text=True)
    assert "reads sorted on the device" in r.stderr
    m = [l for l in r.stderr.split("\n") if "21-mer statistics on the device" in l]
    assert m and int(m[0].split(",")[1].split()[0]) > 100, r.stderr[-600:]       # reads were trimmed
    assert "rough annotation on the device" in r.stderr and "AssignRead pass on the device" in r.stderr
    for suf in SUFFIXES:
        a = open(os.path.join(tmp, "stock" + suf), "rb").read()
        assert len(a) > 0 and a == open(os.path.join(tmp, "dev" + suf), "rb").read(), suf


def test_batch_emu_repseq_and_min_cov(emu_batch_binary, tmp_path):
    run_and_compare(emu_batch_binary, write_inputs(str(tmp_path), 800, 25, 22), str(tmp_path),
                    extra=("--trimLevel", "2", "--skipMateExtension", "--contigMinCov", "2"), env={"T4_STREAMS": "1"})


def test_batch_emu_barcodes(emu_batch_binary, tmp_path):
    run_and_compare(emu_batch_binary, write_barcode_inputs(str(tmp_path)), str(tmp_path), extra=("--contigMinCov", "4"), env={"T4_STREAMS": "1"})


def test_batch_emu_sharded_runs(emu_batch_binary, tmp_path):
    """S > 1: read-sharded assembly (SURVEY.md 8e) through the same driver; the output differs from the unsharded run by
    definition, so only the invariants are checked: it completes, every assembled read is reported once, contigs exist --
    for both stream assignments of t4_shard_reads (T4_SHARD_BY=gene, the default, and rank); grouping by gene must not
    fragment the assembly more than rank blocks do."""
    tmp = str(tmp_path)
    args = write_inputs(tmp, 600, 20, 25)
    n_contigs = {}
    for by in ("gene", "rank"):
        e = dict(os.environ, T4_STREAMS="3", T4_SHARD_BY=by)
        pre = os.path.join(tmp, "s3" + by)
        subprocess.run([emu_batch_binary, "-t", "1", "-o", pre] + args, check=True, stdout=subprocess.DEVNULL,
                       stderr=subprocess.DEVNULL, timeout=900, env=e)
        raw = open(pre + "_raw.out").read()
        names = [l.split()[0] for l in raw.split("\n") if l.startswith(">")]
        assert len(names) > 5 and len(set(names)) == len(names)          # global slot numbers are unique
        reads = [l for l in open(pre + "_assembled_reads.fa") if l.startswith(">")]
        assert len(reads) > 600 and len(set(reads)) == len(reads)
        n_contigs[by] = len(names)
    assert n_contigs["gene"] <= n_contigs["rank"], n_contigs


def test_dropin_emu_shipped_example(emu_binary, tmp_path):
    """BASELINE.json configs[0]: example_1.fq + example_2.fq -f hg38_bcrtcr.fa, -t 1."""
    run_and_compare(emu_binary, example_inputs(str(tmp_path)), str(tmp_path))


def test_dropin_emu_synthetic(emu_binary, tmp_path):
    run_and_compare(emu_binary, write_inputs(str(tmp_path)), str(tmp_path))


def test_dropin_emu_repseq_flags(emu_binary, tmp_path):
    """run-trust4 --repseq expands to --trimLevel 2 --skipMateExtension (run-trust4:288-291): repetitiveData = true."""
    run_and_compare(emu_binary, write_inputs(str(tmp_path), 800, 25, 22), str(tmp_path), extra=("--trimLevel", "2", "--skipMateExtension"))


def test_dropin_emu_contig_min_cov(emu_binary, tmp_path):
    """--contigMinCov: ReleaseShallowContigs before Output (main.cpp:1952-1955) runs on the device set."""
    run_and_compare(emu_binary, write_inputs(str(tmp_path), 800, 25, 24), str(tmp_path), extra=("--contigMinCov", "3"))


@pytest.mark.parametrize("extra", [(), ("--contigMinCov", "4")])
def test_dropin_emu_barcodes(emu_binary, tmp_path, extra):
    """--barcode: hitLenRequired 13, barcode-salted index, ReleaseFinishedBarcodeSeq after a cell's last read
    (main.cpp:1549-1560, 1846-1859), barcode names in Output."""
    run_and_compare(emu_binary, write_barcode_inputs(str(tmp_path)), str(tmp_path), extra=extra)


@pytest.mark.gpu
def test_dropin_gpu_barcodes(tmp_path):
    binary = prebuilt("trust4_gpu")
    run_and_compare(binary, write_barcode_inputs(str(tmp_path)), str(tmp_path), extra=("--contigMinCov", "4"))


@pytest.mark.gpu
def test_batch_gpu_synthetic_and_barcodes(tmp_path):
    binary = prebuilt("trust4_gpu_batch")
    a = tmp_path / "a"
    b = tmp_path / "b"
    a.mkdir()
    b.mkdir()
    run_and_compare(binary, write_inputs(str(a), 3000, 60, 27), str(a), env={"T4_STREAMS": "1"})
    run_and_compare(binary, write_barcode_inputs(str(b)), str(b), extra=("--contigMinCov", "4"), env={"T4_STREAMS": "1"})


@pytest.mark.gpu
def test_dropin_gpu_synthetic(tmp_path):
    binary = prebuilt("trust4_gpu")
    run_and_compare(binary, write_inputs(str(tmp_path)), str(tmp_path))
