"""CPU: the product's host-side eager-output code (libfsm_b200/csrc/eager_host.h -- the initial
partition of fsm_minimise with the reference's blind spot, the per-state id masks of
fsm_b200_dfa_compile), compiled for the CPU by oracle/eager_host_test.cpp and checked against the
compiled reference, live."""
import ctypes as C
import os

import numpy as np
import pytest

import reflib
from libfsm_b200.desc import CDesc, FlatFsm
from test_oracle_determinise import assert_isomorphic
from test_oracle_eager import diamond, random_nfa

SO = os.path.join(reflib.REF_DIR, "libeager_host.so")


@pytest.fixture(scope="module")
def host():
    if not os.path.exists(SO):
        reflib.build_oracle()
    lib = C.CDLL(SO, use_errno=True)
    lib.eager_host_minimise.argtypes = [C.POINTER(CDesc), C.POINTER(reflib.OwnedDesc)]
    lib.eager_host_masks.argtypes = [C.POINTER(CDesc), C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_void_p),
                                     C.POINTER(C.c_void_p)]
    lib.oracle_desc_free.argtypes = [C.POINTER(reflib.OwnedDesc)]
    lib.oracle_desc_free.restype = None
    return lib


def host_minimise(lib, f: FlatFsm) -> FlatFsm:
    od = reflib.OwnedDesc()
    assert lib.eager_host_minimise(C.byref(f.as_c()), C.byref(od)) == 0
    try:
        if od.desc.nstates == 0:
            return None
        return reflib._take_eager(FlatFsm.from_c(od.desc), od.eager_off, od.eager_ids)
    finally:
        lib.oracle_desc_free(C.byref(od))


@pytest.mark.parametrize("eager", [{1: [7]}, {2: [7]}, {1: [7], 2: [7]}, {1: [7], 2: [8]}, {0: [1], 3: [2]}])
def test_initial_partition_quirk_cases(host, oracle, ref, eager):
    f = diamond(eager)
    h = ref.from_flat(f)
    ref.minimise(h)
    want = ref.flatten(h)
    ref.free(h)
    assert_isomorphic(oracle, host_minimise(host, f), want)


@pytest.mark.parametrize("seed", range(80))
def test_initial_partition_random_pipeline(host, oracle, ref, seed):
    rng = np.random.default_rng(7000 + seed)
    nfa = random_nfa(rng, int(rng.integers(3, 20)))
    h = ref.from_flat(nfa)
    ref.determinise(h)
    d_ref = ref.flatten(h)
    ref.minimise(h)
    m_ref = ref.flatten(h)
    ref.free(h)
    got = host_minimise(host, d_ref)
    if m_ref.nstates == 0:
        assert got is None
    else:
        assert_isomorphic(oracle, got, m_ref)


def test_masks_match_the_id_sets(host):
    rng = np.random.default_rng(5)
    f = random_nfa(rng, 12, with_eps=False)
    nbits, ids, masks = C.c_uint32(0), C.c_void_p(), C.c_void_p()
    words = host.eager_host_masks(C.byref(f.as_c()), f.nstates + 1, C.byref(nbits), C.byref(ids), C.byref(masks))
    assert words == (nbits.value + 63) // 64 and nbits.value == len(set(int(x) for x in f.eager_ids))
    idl = np.ctypeslib.as_array(C.cast(ids, C.POINTER(C.c_uint32)), shape=(nbits.value,)).copy()
    m = np.ctypeslib.as_array(C.cast(masks, C.POINTER(C.c_uint64)), shape=(f.nstates + 1, words)).copy()
    assert list(idl) == sorted(set(int(x) for x in f.eager_ids))
    for s in range(f.nstates):
        got = [int(idl[b]) for b in range(nbits.value) if (int(m[s, b >> 6]) >> (b & 63)) & 1]
        assert got == [int(x) for x in f.eager_of(s)]
    assert not m[f.nstates].any()            # the dead row fires nothing
    libc = C.CDLL(None); libc.free.argtypes = [C.c_void_p]
    libc.free(ids); libc.free(masks)
