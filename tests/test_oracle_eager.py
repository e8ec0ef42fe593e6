"""CPU: eager outputs (include/fsm/fsm.h:273-336) -- the oracle restatement against the compiled
reference, live: ids fired by fsm_exec (exec.c:126-144), carried by fsm_determinise over epsilon
closures and member sets (epsilons.c:221-253, determinise.c:2614-2636), separating classes in
fsm_minimise (minimise.c:705-731) -- including the reference's habit of not looking at the eager
ids of states listed behind the first plain state of a class (minimise.c:771-782)."""
import numpy as np
import pytest

import reflib
from libfsm_b200.desc import FlatFsm
from test_oracle_determinise import assert_isomorphic

import os  # noqa: E402
import goldenio  # noqa: E402

GOLDEN = goldenio.load_eager_cases(os.path.join(goldenio.GOLDEN_DIR, "golden_eager.npz"))


@pytest.mark.parametrize("case", GOLDEN, ids=[c["name"] for c in GOLDEN])
def test_oracle_against_recorded_reference(oracle, case):
    """tests/golden/golden_eager.npz (recorded from the reference by make_golden.py eager; no
    reference needed to run): determinise, minimise and the fired id sets of fsm_exec."""
    assert_isomorphic(oracle, oracle.determinise(case["nfa"]), case["dfa"])
    m = oracle.minimise(case["dfa"])
    if case["min"] is None:
        assert m.nstates == 0
        return
    assert_isomorphic(oracle, m, case["min"])
    for s, ids, ret in zip(case["inputs"], case["fired"], case["rets"]):
        rec, got = oracle.exec_eager(case["min"], s)
        assert rec[0] == ret and got == ids, s


def diamond(eager):
    """0 -a-> 1 -c-> 3(end), 0 -b-> 2 -c-> 3: states 1 and 2 are equivalent but for eager ids."""
    return FlatFsm.from_edges(4, 0, [3], [(0, ord("a"), 1), (0, ord("b"), 2), (1, ord("c"), 3), (2, ord("c"), 3)],
                              eager=eager)


@pytest.mark.parametrize("eager,nstates", [({1: [7]}, 3), ({2: [7]}, 4), ({1: [7], 2: [7]}, 3), ({1: [7], 2: [8]}, 4),
                                           ({0: [1], 3: [2]}, 3)])
def test_minimise_quirk_is_the_references(oracle, ref, eager, nstates):
    f = diamond(eager)
    h = ref.from_flat(f)
    ref.minimise(h)
    want = ref.flatten(h)
    ref.free(h)
    assert want.nstates == nstates          # recorded behaviour of the reference, not an opinion
    assert_isomorphic(oracle, oracle.minimise(f), want)


def random_nfa(rng, n, with_eps=True):
    edges = [(int(rng.integers(n)), [97 + int(x) for x in rng.integers(0, 4, size=int(rng.integers(1, 3)))], int(rng.integers(n)))
             for _ in range(int(rng.integers(n, 3 * n)))]
    eps = [(int(rng.integers(n)), int(rng.integers(n))) for _ in range(int(rng.integers(0, n // 2 + 1)))] if with_eps else []
    ends = sorted({int(x) for x in rng.integers(n, size=max(1, n // 3))})
    eager = {int(s): [int(x) for x in rng.integers(1, 6, size=int(rng.integers(1, 3)))]
             for s in rng.integers(n, size=int(rng.integers(1, n // 2 + 2)))}
    endids = {e: [int(x) for x in rng.integers(10, 14, size=int(rng.integers(0, 3)))] for e in ends}
    return FlatFsm.from_edges(n, 0, ends, edges, eps=eps, endids=endids, eager=eager)


@pytest.mark.parametrize("seed", range(60))
def test_pipeline_with_eager_outputs_random(oracle, ref, seed):
    rng = np.random.default_rng(4000 + seed)
    nfa = random_nfa(rng, int(rng.integers(3, 14)))
    h = ref.from_flat(nfa)
    assert ref.flatten(h).eager_ids is not None
    # determinise: same sets, same carried eager ids
    ref.determinise(h)
    d_ref = ref.flatten(h)
    d_orc = oracle.determinise(nfa)
    assert_isomorphic(oracle, d_orc, d_ref)
    # exec on the reference's DFA: records and fired id sets
    al = np.frombuffer(b"abcdx", dtype=np.uint8)
    for _ in range(25):
        s = al[rng.integers(0, al.size, int(rng.integers(0, 8)))].tobytes()
        assert oracle.exec_eager(d_ref, s)[1] == ref.exec_eager(h, s)[1], s
        got, want = oracle.exec_eager(d_ref, s)[0], ref.exec_eager(h, s)[0]
        assert got[0] == want[0] and got[2] == want[2] and (got[0] != 1 or got[1] == want[1])
    # minimise in pipeline order (same struct fsm)
    ref.minimise(h)
    m_ref = ref.flatten(h)
    m_orc = oracle.minimise(d_ref)
    if m_ref.nstates == 0:
        assert m_orc.nstates == 0
    else:
        assert_isomorphic(oracle, m_orc, m_ref)
    ref.free(h)


@pytest.mark.parametrize("patterns,inputs", [
    (["abc", "b+", "xyz"], [b"abc", b"zabcz", b"bbb", b"xyzabc", b"", b"q"]),
    (["^ab", "cd$", "e"], [b"ab", b"xab", b"cd", b"cdx", b"abecd", b"e"]),
])
def test_union_repeated_pattern_group_pipeline(oracle, ref, patterns, inputs):
    """The reference's own producer of eager outputs (tests/eager_output/utils.c:run_test):
    re_comp(RE_SAVE_LINKAGE_INFO) x N -> fsm_union_repeated_pattern_group -> determinise -> minimise
    -> exec with the callback; the oracle must agree at every stage."""
    RE_SAVE_LINKAGE_INFO = 1 << 9      # include/re/re.h:34
    try:
        hs = [ref.re_comp(p, flags=RE_SAVE_LINKAGE_INFO) for p in patterns]
    except ValueError:
        pytest.skip("flag value differs in this reference build")
    u = ref.union_repeated_pattern_group(hs, 1)
    nfa = ref.flatten(u)
    ref.determinise(u)
    d_ref = ref.flatten(u)
    assert_isomorphic(oracle, oracle.determinise(nfa), d_ref)
    ref.minimise(u)
    m_ref = ref.flatten(u)
    assert_isomorphic(oracle, oracle.minimise(d_ref), m_ref)
    for s in inputs:
        assert oracle.exec_eager(m_ref, s)[1] == ref.exec_eager(u, s)[1], s
    ref.free(u)
