"""The reference's DFA state NUMBERING, replayed by the product's refnum.h functions.

libfsm_b200/csrc/refnum.h holds the host+device inline code K2 uses to number DFA states the
way fsm_determinise does (LIFO worklist, determinise.c:118-185, over the entry order of the
pairwise label-group analysis, determinise.c:898-1054 / :1056-1335 / :2331-2505).
oracle/refnum_host.cpp compiles those same functions for the CPU; here their output is compared
BIT-EXACTLY (no canonicalisation) with the DFAs the reference recorded in
tests/golden/golden_determinise.npz and with the reference's runs on random NFAs: live where the
compiled reference is built (table by table), otherwise against the digest of each DFA it recorded.
"""
import ctypes as C
import os

import numpy as np
import pytest

import goldenio
import reflib
from libfsm_b200.desc import CDesc, FlatFsm

SO = os.path.join(reflib.REF_DIR, "librefnum_host.so")


@pytest.fixture(scope="module")
def host():
    if not os.path.exists(SO):
        reflib.build_oracle()
    lib = C.CDLL(SO, use_errno=True)
    lib.refnum_host_determinise.argtypes = [C.POINTER(CDesc), C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_void_p),
                                            C.POINTER(C.c_void_p)]
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]

    def run(f: FlatFsm):
        n, tab, end = C.c_uint32(0), C.c_void_p(), C.c_void_p()
        rc = lib.refnum_host_determinise(C.byref(f.as_c()), 200000, C.byref(n), C.byref(tab), C.byref(end))
        assert rc == 0
        D = n.value
        if D == 0:
            return np.zeros((0, 256), np.uint32), np.zeros(0, np.uint8)
        t = np.ctypeslib.as_array(C.cast(tab, C.POINTER(C.c_uint32)), shape=(D, 256)).copy()
        e = np.ctypeslib.as_array(C.cast(end, C.POINTER(C.c_uint8)), shape=(D,)).copy()
        libc.free(tab); libc.free(end)
        return t, e
    return run


def assert_numbering(ref, h, table: np.ndarray, end: np.ndarray, note=None) -> None:
    """The host's DFA equals the reference's DFA behind h, state numbering included.  Against the live
    reference the tables are compared row by row first, so that a failure names the states that differ."""
    if isinstance(ref, reflib.Ref):
        dfa = ref.flatten(h)
        assert table.shape[0] == dfa.nstates, (note, table.shape[0], dfa.nstates)
        bad = np.nonzero((table != dfa.dense_table()).any(axis=1) | (end.astype(bool) != np.asarray(dfa.is_end).astype(bool)))[0]
        assert bad.size == 0, (note, "states numbered differently from the reference's:", bad[:10])
    assert reflib.numbering_digest(table, end) == ref.numbering(h), (note, "state numbering differs from the reference's")


DET_CASES = goldenio.load_det_cases(os.path.join(goldenio.GOLDEN_DIR, "golden_determinise.npz"))


@pytest.mark.parametrize("case", DET_CASES, ids=[c["name"] for c in DET_CASES])
def test_numbering_matches_recorded_reference(host, case):
    nfa, dfa = case["nfa"], case["dfa"]
    if not nfa.hasstart:
        pytest.skip("no start state: fsm_determinise leaves the fsm as is")
    table, end = host(nfa)
    assert table.shape[0] == dfa.nstates
    assert np.array_equal(table, dfa.dense_table()), "state numbering differs from the reference's"
    assert np.array_equal(end.astype(bool), np.asarray(dfa.is_end).astype(bool))


def _random_nfa(rng, n, nedges, neps, nsyms):
    edges = []
    for _ in range(nedges):
        a, b = int(rng.integers(n)), int(rng.integers(n))
        lo = int(rng.integers(nsyms))
        hi = min(nsyms, lo + 1 + int(rng.integers(4)))
        edges.append((a, list(range(97 + lo, 97 + hi)), b))
    eps = [(int(rng.integers(n)), int(rng.integers(n))) for _ in range(neps)]
    ends = sorted({int(x) for x in rng.integers(n, size=max(1, n // 4))})
    return FlatFsm.from_edges(n, 0, ends, edges, eps=eps)


@pytest.mark.parametrize("seed", range(40))
def test_numbering_matches_live_reference_random(host, seed):
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(2, 40))
    nfa = _random_nfa(rng, n, int(rng.integers(1, 4 * n)), int(rng.integers(0, n)), int(rng.integers(1, 9)))
    ref = reflib.reference()
    h = ref.from_flat(nfa)
    ref.determinise(h)
    assert_numbering(ref, h, *host(nfa))
    ref.free(h)


@pytest.mark.parametrize("words,length", [(50, 12), (300, 30)])
def test_numbering_matches_live_reference_config5_shape(host, words, length):
    from libfsm_b200 import workloads
    nfa = workloads.config5_nfa(words, length)
    ref = reflib.reference()
    h = ref.from_flat(nfa)
    ref.determinise(h)
    assert_numbering(ref, h, *host(nfa))
    ref.free(h)


try:
    from hypothesis import HealthCheck, given, settings, strategies as st
    from test_oracle_property import regex as _regex
except ImportError:                                   # hypothesis is optional
    _regex = None

if _regex is not None:
    @settings(max_examples=80, deadline=None, derandomize=reflib.REF_MODE == "record" or reflib.replaying(), suppress_health_check=[HealthCheck.function_scoped_fixture, HealthCheck.too_slow])
    @given(patterns=st.lists(_regex, min_size=1, max_size=4))
    def test_numbering_matches_live_reference_regex_unions(host, patterns):
        """ε-heavy NFAs the way re(1)/rx(1) build them: re_comp, end ids, fsm_union_array
        (3000 examples of this strategy were run once while pinning; 80 per suite run)."""
        ref = reflib.reference()
        hs = []
        try:
            for p in patterns:
                hs.append(ref.re_comp(p))
        except ValueError:
            for h in hs:
                ref.free(h)
            return
        if len(hs) > 1:
            for i, h in enumerate(hs):
                ref.setendid(h, i + 1)
            u = ref.union_array(hs)
        else:
            u = hs[0]
        nfa = ref.flatten(u)
        ref.determinise(u)
        assert_numbering(ref, u, *host(nfa), note=patterns)
        ref.free(u)
