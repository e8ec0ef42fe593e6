"""CPU: the DFAVM bytecode loader (fsm_b200_dfavm_load; SURVEY.md section 8(f)4) against images written by
the reference itself (fsm_vm_compile + fsm_dfavm_save through oracle/ref_harness.c): the loaded automaton
must be a DFA and give, on the golden inputs, the verdicts the reference's fsm_exec recorded AND the
verdicts its own bytecode interpreter (fsm_vm_match_buffer) gives."""
import errno
import os

import numpy as np
import pytest

import goldenio
import reflib
import libfsm_b200 as L

CASES = [c for c in goldenio.load_exec_cases(os.path.join(goldenio.GOLDEN_DIR, "golden_exec.npz")) if c["is_dfa"]]


@pytest.mark.parametrize("case", CASES[::2], ids=lambda c: c["name"])
def test_loaded_image_matches_like_the_reference(ref, oracle, case):
    h = ref.from_flat(case["fsm"])
    image = ref.dfavm_bytes(h)
    vm = ref.vm_match_batch(h, case["base"], case["offsets"], nthreads=2)
    ref.free(h)
    assert image[:8] == b"DFAVM$\x00\x01"
    f = L.load_dfavm(image)
    assert oracle.isdfa(f) and f.hasstart
    got = oracle.exec_batch(f, case["base"], case["offsets"])
    assert (got["ret"] == case["expect"]["ret"]).all(), case["name"]
    assert ((got["ret"] == 1) == (vm == 1)).all()
    L.plan(f)                                   # and the engine lays it out like any other DFA


def test_malformed_images_are_refused():
    with pytest.raises(L.FsmB200Error) as e:
        L.load_dfavm(b"not a dfavm image....")
    assert e.value.errno == errno.EINVAL
    with pytest.raises(L.FsmB200Error) as e:
        L.load_dfavm(b"DFAVM$\x00\x02" + (4).to_bytes(4, "little") + b"\x08\x00\x00\x00")
    assert e.value.errno == errno.ENOTSUP
    with pytest.raises(L.FsmB200Error) as e:
        L.load_dfavm(b"DFAVM$\x00\x01" + (100).to_bytes(4, "little") + b"\x08")
    assert e.value.errno == errno.EINVAL
