"""CPU: differential of the oracle restatement against the compiled reference
(oracle/_ref/libref_harness.so), or against its recorded answers where it is not built."""
import zlib

import numpy as np
import pytest

import reflib

PATTERNS = [r"a[ -~]{7}\z", r"[0-9]+\.[0-9]+", r"^abc[0-9]+x$", r"(foo|bar)+baz", r"^$", r"a*b*c*",
            r"^[a-z]+@[a-z]+\.(com|org)$", r"x{3,5}y", r"(?i)hello", r"[^a]b"]


@pytest.mark.parametrize("pattern", PATTERNS)
def test_exec_random_inputs(oracle, ref, pattern):
    h = ref.compile_dfa(pattern)
    f = ref.flatten(h)
    rng = np.random.default_rng(zlib.crc32(pattern.encode()))
    alpha = np.frombuffer(b"abcxyz0123456789.@fobarhelHELO \n\x00", dtype=np.uint8)
    strs = [alpha[rng.integers(0, len(alpha), int(rng.integers(0, 64)))].tobytes() for _ in range(2000)]
    base, off = reflib.offsets_for(strs)
    got = oracle.exec_batch(f, base, off)
    exp0 = ref.exec_batch(h, base, off, mode=0)
    exp1 = ref.exec_batch(h, base, off, mode=1)
    assert (got["ret"] == exp0["ret"]).all() and (got["consumed"] == exp0["consumed"]).all()
    assert (got["end"][exp0["ret"] == 1] == exp0["end"][exp0["ret"] == 1]).all()
    assert (got == exp1).all()
    ref.free(h)


def test_round_trip_desc(oracle, ref):
    """flatten -> refh_from_desc -> flatten is the identity, and fsm_equal agrees."""
    h = ref.compile_dfa(r"(ab|cd)*e")
    f = ref.flatten(h)
    h2 = ref.from_flat(f)
    f2 = ref.flatten(h2)
    assert ref.equal(h, h2)
    assert (f.dense_table() == f2.dense_table()).all() and (f.is_end == f2.is_end).all()
    ref.free(h); ref.free(h2)


def test_nfa_rejected_like_reference(oracle, ref):
    h = ref.re_comp(r"ab*c|abd")
    f = ref.flatten(h)
    assert ref.exec(h, b"abc")[0] == -1
    assert oracle.exec(f, b"abc")[0] == -1
    ref.free(h)


def test_endids_match_reference(oracle, ref):
    hs = []
    for i, p in enumerate(["abc", "def", "abc.def"]):
        hh = ref.compile_dfa(p)
        ref.setendid(hh, 10 + i)
        hs.append(hh)
    u = ref.union_array(hs)
    ref.determinise(u)
    f = ref.flatten(u)
    for s in (b"abc", b"abcxdef", b"def", b"zzz"):
        rc, end, _ = ref.exec(u, s)
        ret, oend, _ = oracle.exec(f, s)
        assert rc == ret
        if rc == 1:
            assert end == oend
            assert list(f.endids_of(end)) == ref.endids(u, end)
    ref.free(u)


def test_config4_validator_is_utf8dfa_starred(ref, oracle):
    """BASELINE config 4's DFA: golden_cfg4.npz holds examples/utf8dfa (0..10FFFF, 9 states for one code
    point) starred through the reference API, det + min (8 states); its meta records fsm_equal with the
    PCRE-built validator of golden_exec.npz.  Live here: the same construction on 0..7FF must agree
    with the full-range validator on 1- and 2-byte text, and the fixture equals the PCRE automaton."""
    import os
    import numpy as np
    import goldenio
    g = goldenio.load_cfg4()
    assert g["meta"]["one_codepoint_states"] == 9 and g["meta"]["validator_states"] == 8 and g["meta"]["fsm_equal"] is True
    cases = {c["name"]: c for c in goldenio.load_exec_cases(os.path.join(goldenio.GOLDEN_DIR, "golden_exec.npz"))}
    pcre = cases[g["meta"]["fsm_equal_with"]]
    a, b = ref.from_flat(g["fsm"]), ref.from_flat(pcre["fsm"])
    assert ref.equal(a, b)
    ref.free(a); ref.free(b)
    # the recorded reference answers of the PCRE-built validator hold for the utf8dfa-built one
    got = oracle.exec_batch(g["fsm"], pcre["base"], pcre["offsets"])
    assert (got["ret"] == pcre["expect"]["ret"]).all() and (got["consumed"] == pcre["expect_amortised"]["consumed"]).all()
    h = ref.utf8dfa(0, 0x7FF)
    assert ref.countstates(h) == 3
    ref.star(h); ref.determinise(h); ref.minimise(h)
    small = ref.flatten(h)
    ref.free(h)
    from libfsm_b200 import workloads
    text = workloads.utf8_host(20000, seed=5)
    text = text[text < 0xE0]                     # keep 1- and 2-byte sequences only ... and re-validate below
    full = oracle.exec(g["fsm"], text.tobytes(), validate=False)
    part = oracle.exec(small, text.tobytes(), validate=False)
    assert full[0] == part[0] and full[2] == part[2]
