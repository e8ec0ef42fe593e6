"""GPU: eager outputs (include/fsm/fsm.h:273-336; SURVEY.md section 8(f)2) through the engine and
through the shim.

Status: the semantics are pinned on the CPU -- the oracle against the live reference
(tests/test_oracle_eager.py), the product's host-side code against the reference
(tests/test_eager_host.py), and the whole shim with the reference's 22 tests/eager_output programs
over the CPU stub engine (tests/test_shim_hostlogic.py).  The CUDA side (k1_eager.cu, the carry in
K2/K3) passed on the driver's B200 at the end of round 1; plain (strict) tests since round 2.
"""
import os
import subprocess

import numpy as np
import pytest

import reflib
import libfsm_b200 as L
from test_oracle_determinise import assert_isomorphic
from test_oracle_eager import diamond, random_nfa

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFTESTS_DIR = os.path.join(ROOT, "build", "shim", "reftests")
EAGER_PROGRAMS = sorted(x for x in os.listdir(REFTESTS_DIR) if x.startswith("eager_output")) if os.path.isdir(REFTESTS_DIR) else []


import goldenio  # noqa: E402

GOLDEN = goldenio.load_eager_cases(os.path.join(goldenio.GOLDEN_DIR, "golden_eager.npz"))


@pytest.mark.parametrize("case", GOLDEN, ids=[c["name"] for c in GOLDEN])
def test_against_recorded_reference(oracle, case):
    """tests/golden/golden_eager.npz: what the reference itself produced -- determinise (K2),
    minimise (K3) compared in canonical form incl. the eager-id sets, fsm_exec's fired ids
    (k1_eager.cu) compared as sets."""
    assert_isomorphic(oracle, L.determinise(case["nfa"]), case["dfa"])
    m = L.minimise(case["dfa"])
    if case["min"] is None:
        assert m.nstates == 0
        return
    assert_isomorphic(oracle, m, case["min"])
    base, off = reflib.offsets_for(case["inputs"])
    with L.Dfa(case["min"]) as dfa:
        if len(dfa.eager_ids()) == 0:
            return
        rec, masks = dfa.exec_batch_eager(base, off)
        got = [dfa.fired_ids(masks[i]) for i in range(len(case["inputs"]))]     # decode while the DFA is alive
    for i, (ids, ret) in enumerate(zip(case["fired"], case["rets"])):
        assert int(rec["ret"][i]) == ret
        assert got[i] == ids, case["inputs"][i]


@pytest.mark.parametrize("seed", range(12))
def test_exec_fired_sets_match_the_oracle(oracle, seed):
    rng = np.random.default_rng(8100 + seed)
    nfa = random_nfa(rng, int(rng.integers(4, 16)))
    dfa_desc = oracle.determinise(nfa)
    if dfa_desc.eager_ids is None:
        pytest.skip("no eager output on a reachable state of this automaton")
    al = np.frombuffer(b"abcdx", dtype=np.uint8)
    strs = [al[rng.integers(0, al.size, int(rng.integers(0, 40)))].tobytes() for _ in range(500)] + [b""]
    base, off = reflib.offsets_for(strs)
    with L.Dfa(dfa_desc) as dfa:
        assert list(dfa.eager_ids()) == sorted(set(int(x) for x in dfa_desc.eager_ids))
        rec, masks = dfa.exec_batch_eager(base, off)
        plain = dfa.exec_batch(base, off)             # the plain entry points work on such a DFA too
        fired = [dfa.fired_ids(masks[i]) for i in range(len(strs))]
    assert (rec == plain).all()
    for i, s in enumerate(strs):
        want_rec, want_ids = oracle.exec_eager(dfa_desc, s)
        assert (int(rec["ret"][i]), int(rec["consumed"][i])) == (want_rec[0], want_rec[2]), s
        if want_rec[0] == 1:
            assert int(rec["end"][i]) == want_rec[1]
        assert fired[i] == want_ids, s


@pytest.mark.parametrize("seed", range(12))
def test_determinise_and_minimise_carry_eager_outputs(oracle, seed):
    rng = np.random.default_rng(8200 + seed)
    nfa = random_nfa(rng, int(rng.integers(4, 20)))
    d = L.determinise(nfa)
    assert_isomorphic(oracle, d, oracle.determinise(nfa))
    m = L.minimise(d)
    want = oracle.minimise(d)
    if want.nstates == 0:
        assert m.nstates == 0
    else:
        assert_isomorphic(oracle, m, want)


@pytest.mark.parametrize("eager", [{1: [7]}, {2: [7]}, {1: [7], 2: [8]}])
def test_minimise_blind_spot_like_the_reference(oracle, eager):
    f = diamond(eager)
    assert_isomorphic(oracle, L.minimise(f), oracle.minimise(f))


@pytest.mark.skipif(not EAGER_PROGRAMS, reason="reference eager_output tests not built against the shim")
@pytest.mark.parametrize("name", EAGER_PROGRAMS)
def test_reference_eager_output_programs_against_the_shim(name):
    """tests/eager_output/*.c of the reference, unmodified: re_comp x N ->
    fsm_union_repeated_pattern_group -> fsm_determinise (K2) -> fsm_minimise (K3) -> fsm_exec with
    the callback (k1_eager.cu)."""
    p = subprocess.run([os.path.join(REFTESTS_DIR, name)], capture_output=True, timeout=300)
    assert p.returncode == 0, (name, p.stdout.decode()[-2000:], p.stderr.decode()[-2000:])


def test_eager_selftest_program_against_the_shim():
    """libfsm_b200/shim/shim_eager_selftest.c linked to the shim and the CUDA engine: fsm_exec with
    the callback and fsm_exec_batch_eager agree and give the expected id sets."""
    exe = os.path.join(ROOT, "build", "shim", "shim_eager_selftest")
    if not os.path.exists(exe):
        pytest.skip("shim_eager_selftest not built")
    p = subprocess.run([exe], capture_output=True, timeout=300)
    assert p.returncode == 0, (p.stdout.decode(), p.stderr.decode())


def test_one_long_input_with_eager_outputs_is_chunked_and_exact(ref):
    """fsm_exec on ONE long input of an automaton with eager outputs (what the shim calls for it): K1b's
    chunk maps give every chunk's true entry state, the lines kernel walks the chunks from those states and
    the per-chunk id sets are OR-ed -- record and id set equal the reference's single serial walk, through
    the host and the device entry point, and it is not one lane (several launches)."""
    import torch
    from libfsm_b200 import workloads
    c = goldenio.load_cfg3()["eager"]
    _, inst = workloads.cfg3_patterns()
    base, _ = workloads.cfg3_lines_host(60000, inst, seed=33)
    h = ref.from_flat(c["fsm"])
    cuts = (8 << 20, (3 << 20) + 17, (1 << 21) + 5)
    wants = [ref.exec_eager_batch(h, np.ascontiguousarray(base[:cut]), np.array([0, cut], dtype=np.uint64), c["idlist"],
                                  mode=1, nthreads=1) for cut in cuts]
    ref.free(h)
    with L.Dfa(c["fsm"]) as dfa:
        for cut, (want, wmasks) in zip(cuts, wants):
            data = np.ascontiguousarray(base[:cut])
            off = np.array([0, cut], dtype=np.uint64)
            L.launch_count(reset=True)
            rec, masks = dfa.exec_batch_eager(data, off)
            assert L.launch_count() >= 5, "expected the chunked path"
            assert (rec == want).all() and (masks == wmasks).all(), cut
            drec, dmasks = dfa.exec_batch_eager(torch.from_numpy(data).cuda(), torch.from_numpy(off.astype(np.int64)).cuda())
            torch.cuda.synchronize()
            assert (L.results_from_torch(drec) == want).all() and (dmasks.cpu().numpy().view(np.uint64) == wmasks).all(), cut
        # fewer ids fire on a prefix: the OR really is over the chunks walked
        assert (wmasks != 0).any()


@pytest.mark.parametrize("die_at", [None, 100, 70000, 299999])
def test_one_long_input_eager_with_a_missing_edge(oracle, die_at):
    """The same path on a small INCOMPLETE automaton with eager outputs: the walk dies in a prefix window
    or in a chunk body; ids fired before the missing edge count, nothing after it does."""
    rng = np.random.default_rng(8100)
    dfa_desc = None
    for seed in range(40):
        nfa = random_nfa(np.random.default_rng(8200 + seed), 12)
        d = oracle.determinise(nfa)
        if d.eager_ids is not None and d.nstates >= 4:
            dfa_desc = d
            break
    assert dfa_desc is not None
    al = np.frombuffer(b"abcd", dtype=np.uint8)
    # a long input that stays alive: walk the oracle greedily over bytes that have an edge
    tab = oracle.flatten(dfa_desc)
    st, out = dfa_desc.start, []
    for _ in range(300000):
        ok = [b for b in al if tab[st, b] != 0xFFFFFFFF]
        if not ok:
            break
        b = int(ok[int(rng.integers(len(ok)))]); out.append(b); st = int(tab[st, b])
    data = np.array(out, dtype=np.uint8)
    if data.size < 200000:
        pytest.skip("this automaton cannot be kept alive for long")
    if die_at is not None and die_at < data.size:
        data[die_at] = ord("x")                                  # no edge on 'x' anywhere
    want_rec, want_ids = oracle.exec_eager(dfa_desc, data.tobytes())
    off = np.array([0, data.size], dtype=np.uint64)
    with L.Dfa(dfa_desc) as dfa:
        rec, masks = dfa.exec_batch_eager(data, off)
        assert (int(rec["ret"][0]), int(rec["consumed"][0])) == (want_rec[0], want_rec[2])
        assert dfa.fired_ids(masks[0]) == want_ids
