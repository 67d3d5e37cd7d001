"""The C-ABI library loads and exports every symbol include/trust4_b200.h declares (no compute without a GPU)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "trust4_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(t4_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported():
    lib_path = os.path.join(ROOT, "trust4_b200", "libtrust4_b200.so")
    if not os.path.exists(lib_path):
        import __graft_entry__ as ge
        ge.build_lib()
    dll = ctypes.CDLL(lib_path)
    syms = declared_symbols()
    assert len(syms) >= 35
    missing = [s for s in syms if not hasattr(dll, s)]
    assert not missing, missing


def test_python_mirror_covers_header():
    from trust4_b200 import api
    declared = {s[3:] for s in declared_symbols()}
    assert declared == set(api.EXPORTS), declared ^ set(api.EXPORTS)


def test_no_gpu_fails_loudly():
    """Without a CUDA device the product must refuse to work (no CPU fallback)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from trust4_b200 import api
    lib = api.Lib()
    assert lib.init(0, 1 << 20) == api.T4_E_NODEVICE
    assert not lib.seqset_create(9)
    assert b"no CPU fallback" in lib.last_error()


def test_host_utilities_match_reference(ref):
    """t4_has_motif / t4_reverse_complement_in_place are host utilities: callable without a GPU."""
    import numpy as np
    from trust4_b200 import api
    lib = api.Lib()
    r = ref.RefSeqSet(9)
    rng = np.random.default_rng(3)
    for i in range(200):
        s = "".join("ACGTN"[c] for c in rng.choice(5, size=int(rng.integers(5, 160)), p=[.245, .245, .245, .245, .02]))
        for strand in (-1, 0, 1):
            assert lib.has_motif(s.encode(), strand) == r.has_motif(s, strand)
        b = ctypes.create_string_buffer(s.encode())
        lib.reverse_complement_in_place(b, len(s))
        assert b.value.decode() == ref.reverse_complement(s)


def test_lis_matches_reference(ref):
    """t4_test_lis (host utility): the chain rule of the stage-0 scan -- SeqSet::LongestIncreasingSubsequence with its
    tie rules (closest to the average diagonal among equal read offsets, one element per gene offset, the replacement
    sweep) -- on random windows with many ties, against the reference's own member function."""
    import numpy as np
    from trust4_b200 import api
    lib = api.Lib()
    rng = np.random.default_rng(17)
    n_cases = 0
    for it in range(3000):
        n = int(rng.integers(1, 60))
        mode = it % 4
        if mode == 0:      # one diagonal with noise
            b = np.sort(rng.integers(0, 80, size=n))
            a = b + 20 + rng.integers(-10, 11, size=n)
        elif mode == 1:    # heavy ties in both coordinates
            b = np.sort(rng.integers(0, 12, size=n))
            a = rng.integers(0, 12, size=n)
        elif mode == 2:    # two diagonals
            b = np.sort(rng.integers(0, 100, size=n))
            a = b + np.where(rng.random(n) < 0.5, 5, 12)
        else:              # random
            b = np.sort(rng.integers(0, 300, size=n))
            a = rng.integers(0, 300, size=n)
        order = np.lexsort((a, b))             # CompSortPairBInc: b, then a
        a = np.ascontiguousarray(a[order], dtype=np.int32)
        b = np.ascontiguousarray(b[order], dtype=np.int32)
        ga, gb = np.zeros(n, dtype=np.int32), np.zeros(n, dtype=np.int32)
        gl = lib.test_lis(a.ctypes.data, b.ctypes.data, n, ga.ctypes.data, gb.ctypes.data)
        ra, rb = ref.lis(a, b)
        assert gl == len(ra), (it, n, gl, len(ra))
        assert (ga[:gl] == ra).all() and (gb[:gl] == rb).all(), (it, a.tolist(), b.tolist(), ga[:gl].tolist(), ra)
        n_cases += 1
    assert n_cases == 3000
