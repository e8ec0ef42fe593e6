"""CPU: property-based differential pinning of the oracle against the compiled reference:
random regular expressions -> the reference's re_comp NFA -> determinise / minimise / exec by
BOTH the reference and the oracle restatement; DFAs compared in canonical form, exec records
bit for bit."""
import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

import reflib
from test_oracle_determinise import assert_isomorphic

atoms = st.sampled_from(["a", "b", "c", ".", "[ab]", "[^a]", "ab", "(a|b)", r"\d", "x?"])
suffix = st.sampled_from(["", "*", "+", "?", "{1,2}"])
piece = st.builds(lambda a, s: a + s if not (a.endswith("?") and s) else a, atoms, suffix)
branch = st.lists(piece, min_size=1, max_size=4).map("".join)
regex = st.builds(lambda bs, anchor_l, anchor_r: ("^" if anchor_l else "") + "|".join(bs) + ("$" if anchor_r and len(bs) == 1 else ""),
                  st.lists(branch, min_size=1, max_size=3), st.booleans(), st.booleans())


@pytest.mark.needs_ref
@settings(max_examples=60, deadline=None, derandomize=reflib.REF_MODE == "record" or reflib.replaying(), suppress_health_check=[HealthCheck.function_scoped_fixture, HealthCheck.too_slow])
@given(pattern=regex, seed=st.integers(0, 2 ** 31 - 1))
def test_random_regex_pipeline(oracle, ref, pattern, seed):
    try:
        h = ref.re_comp(pattern)
    except ValueError:
        return
    nfa = ref.flatten(h)
    # determinise
    ref.determinise(h)
    d_ref = ref.flatten(h)
    d_orc = oracle.determinise(nfa)
    assert_isomorphic(oracle, d_orc, d_ref)
    # minimise (reference pipeline order: same struct fsm)
    ref.minimise(h)
    m_ref = ref.flatten(h)
    m_orc = oracle.minimise(d_ref)
    if m_ref.nstates == 0:
        assert m_orc.nstates == 0
    else:
        assert_isomorphic(oracle, m_orc, m_ref)
        # exec on the reference's minimised DFA: oracle records == reference records
        rng = np.random.default_rng(seed)
        al = np.frombuffer(b"abcx019 ", dtype=np.uint8)
        strs = [al[rng.integers(0, al.size, int(rng.integers(0, 10)))].tobytes() for _ in range(60)] + [b""]
        base, off = reflib.offsets_for(strs)
        assert (oracle.exec_batch(m_ref, base, off) == ref.exec_batch(h, base, off, mode=1)).all()
        asis = ref.exec_batch(h, base, off, mode=0)
        got = oracle.exec_batch(m_ref, base, off)
        assert (got["ret"] == asis["ret"]).all() and (got["consumed"] == asis["consumed"]).all()
    ref.free(h)
