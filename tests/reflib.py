"""Test-side ctypes wrappers for the two checkers (TEST INFRASTRUCTURE ONLY):

  Oracle  oracle/_ref/libfsm_oracle.so   plain-C restatement (oracle/fsm_oracle.c)
  Ref     oracle/_ref/libref_harness.so  the unmodified reference compiled from
                                         its sources (oracle/ref_harness.c)

Both are built by `make -C oracle`, the harness only where the reference's sources are
present; elsewhere RecordedRef answers with what the harness recorded.  The reference's
sources are never read at test time.
"""
from __future__ import annotations

import atexit
import base64
import ctypes as C
import hashlib
import json
import lzma
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from libfsm_b200.desc import CDesc, CResult, FlatFsm, RESULT_DTYPE  # noqa: E402

REF_DIR = os.path.join(ROOT, "oracle", "_ref")
ORACLE_SO = os.path.join(REF_DIR, "libfsm_oracle.so")
HARNESS_SO = os.path.join(REF_DIR, "libref_harness.so")

RE_LIKE, RE_LITERAL, RE_GLOB, RE_NATIVE, RE_SQL, RE_PCRE = range(6)


def build_oracle() -> None:
    """(Re)build the checkers; builds the reference too when its sources are present."""
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "-j8"], check=True,
                   stdout=subprocess.DEVNULL)


def have_ref() -> bool:
    return os.path.exists(HARNESS_SO)


class OwnedDesc(C.Structure):
    _fields_ = [("desc", CDesc), ("blocks", C.c_void_p * 8), ("eager_off", C.c_void_p), ("eager_ids", C.c_void_p)]


def _take_eager(f: FlatFsm, off_p, ids_p) -> FlatFsm:
    """Attach the eager-output CSR found at (off_p, ids_p) -- C pointers, may be NULL -- to f."""
    if off_p and f.nstates > 0:
        eo = np.ctypeslib.as_array(C.cast(off_p, C.POINTER(C.c_uint64)), shape=(f.nstates + 1,)).copy()
        if int(eo[-1]) > 0:
            f.eager_off = eo
            f.eager_ids = np.ctypeslib.as_array(C.cast(ids_p, C.POINTER(C.c_uint32)), shape=(int(eo[-1]),)).copy()
    return f


def offsets_for(strings) -> tuple[np.ndarray, np.ndarray]:
    """Concatenate byte strings -> (base uint8, offsets uint64[n+1])."""
    lens = np.fromiter((len(s) for s in strings), dtype=np.uint64, count=len(strings))
    offsets = np.zeros(len(strings) + 1, dtype=np.uint64)
    np.cumsum(lens, out=offsets[1:])
    base = np.frombuffer(b"".join(strings), dtype=np.uint8).copy() if len(strings) else np.zeros(0, np.uint8)
    return base, offsets


def _ptr(a: np.ndarray) -> int:
    return a.ctypes.data if a.size else np.zeros(16, dtype=a.dtype).ctypes.data


class Oracle:
    def __init__(self):
        if not os.path.exists(ORACLE_SO):
            build_oracle()
        self.lib = C.CDLL(ORACLE_SO, use_errno=True)
        L, vp, P = self.lib, C.c_void_p, C.POINTER
        L.oracle_isdfa.argtypes = [P(CDesc)]
        L.oracle_exec.argtypes = [P(CDesc), vp, C.c_uint64, C.c_int, P(CResult)]
        L.oracle_exec_batch.argtypes = [P(CDesc), vp, vp, C.c_size_t, C.c_int, C.c_int, vp]
        L.oracle_flatten.argtypes = [P(CDesc), vp]
        L.oracle_flatten.restype = None
        L.oracle_epsilon_closure.argtypes = [P(CDesc), P(vp), P(vp)]
        L.oracle_determinise.argtypes = [P(CDesc), C.c_size_t, P(OwnedDesc)]
        L.oracle_minimise.argtypes = [P(CDesc), P(OwnedDesc)]
        L.oracle_exec_eager.argtypes = [P(CDesc), vp, C.c_uint64, P(CResult), vp, C.c_size_t, P(C.c_size_t)]
        L.oracle_desc_free.argtypes = [P(OwnedDesc)]
        L.oracle_desc_free.restype = None
        L.oracle_canonicalise.argtypes = [P(CDesc), vp, vp]
        L.oracle_canonicalise.restype = C.c_uint32
        self.libc = C.CDLL(None)
        self.libc.free.argtypes = [vp]

    def isdfa(self, f: FlatFsm) -> bool:
        d = f.as_c()
        return bool(self.lib.oracle_isdfa(C.byref(d)))

    def exec(self, f: FlatFsm, data: bytes, validate: bool = True):
        d = f.as_c()
        buf = np.frombuffer(data, dtype=np.uint8) if len(data) else np.zeros(0, np.uint8)
        r = CResult()
        rc = self.lib.oracle_exec(C.byref(d), _ptr(buf), len(data), int(validate), C.byref(r))
        if rc < 0:
            return -1, None, None
        return int(r.ret), int(r.end), int(r.consumed)

    def exec_batch(self, f: FlatFsm, base: np.ndarray, offsets: np.ndarray, nthreads: int = 1,
                   validate_each: bool = False) -> np.ndarray:
        d = f.as_c()
        n = offsets.shape[0] - 1
        out = np.zeros(n, dtype=RESULT_DTYPE)
        rc = self.lib.oracle_exec_batch(C.byref(d), _ptr(base), offsets.ctypes.data, n,
                                        int(validate_each), nthreads, _ptr(out))
        if rc != 0:
            raise OSError(C.get_errno(), "oracle_exec_batch")
        return out

    def flatten(self, f: FlatFsm) -> np.ndarray:
        d = f.as_c()
        t = np.empty((f.nstates, 256), dtype=np.uint32)
        self.lib.oracle_flatten(C.byref(d), _ptr(t))
        return t

    def epsilon_closure(self, f: FlatFsm):
        d = f.as_c()
        off, to = C.c_void_p(), C.c_void_p()
        rc = self.lib.oracle_epsilon_closure(C.byref(d), C.byref(off), C.byref(to))
        assert rc == 0
        o = np.frombuffer((C.c_uint64 * (f.nstates + 1)).from_address(off.value), dtype=np.uint64).copy()
        t = np.frombuffer((C.c_uint32 * max(int(o[-1]), 1)).from_address(to.value), dtype=np.uint32)[:int(o[-1])].copy()
        self.libc.free(off); self.libc.free(to)
        return o, t

    def determinise(self, f: FlatFsm, state_limit: int = 0):
        """-> FlatFsm, or None when the state limit was reached."""
        d = f.as_c()
        od = OwnedDesc()
        rc = self.lib.oracle_determinise(C.byref(d), state_limit, C.byref(od))
        if rc == 1:
            return None
        if rc != 0:
            raise OSError(C.get_errno(), "oracle_determinise")
        try:
            if od.desc.nstates == 0 and not od.desc.group_off:
                return FlatFsm(0, 0, False, np.zeros(0, np.uint8), np.zeros(1, np.uint64),
                               np.zeros((0, 4), np.uint64), np.zeros(0, np.uint32), None, None, None, None)
            return _take_eager(FlatFsm.from_c(od.desc), od.eager_off, od.eager_ids)
        finally:
            self.lib.oracle_desc_free(C.byref(od))

    def exec_eager(self, f: FlatFsm, data: bytes):
        """(record, sorted fired eager-output ids) of one fsm_exec (oracle_exec_eager)."""
        d = f.as_c()
        buf = np.frombuffer(data, dtype=np.uint8)
        r = CResult()
        fired = np.zeros(256, dtype=np.uint32)
        n = C.c_size_t(0)
        ret = self.lib.oracle_exec_eager(C.byref(d), _ptr(buf), len(data), C.byref(r), _ptr(fired), fired.size, C.byref(n))
        assert ret >= 0 and n.value <= fired.size
        return (r.ret, r.end, r.consumed), [int(x) for x in fired[:n.value]]

    def minimise(self, f: FlatFsm) -> FlatFsm:
        d = f.as_c()
        od = OwnedDesc()
        rc = self.lib.oracle_minimise(C.byref(d), C.byref(od))
        if rc != 0:
            raise OSError(C.get_errno(), "oracle_minimise")
        try:
            if od.desc.nstates == 0:
                return FlatFsm(0, 0, False, np.zeros(0, np.uint8), np.zeros(1, np.uint64),
                               np.zeros((0, 4), np.uint64), np.zeros(0, np.uint32), None, None, None, None)
            return _take_eager(FlatFsm.from_c(od.desc), od.eager_off, od.eager_ids)
        finally:
            self.lib.oracle_desc_free(C.byref(od))

    def canonicalise(self, f: FlatFsm):
        """-> (canon_table [ncanon,256], canon_of_state [nstates]) or None if not a DFA."""
        d = f.as_c()
        tab = np.empty((max(f.nstates, 1), 256), dtype=np.uint32)
        cos = np.empty(max(f.nstates, 1), dtype=np.uint32)
        n = self.lib.oracle_canonicalise(C.byref(d), tab.ctypes.data, cos.ctypes.data)
        if n == 0xFFFFFFFF:
            return None
        return tab[:n].copy(), cos[:f.nstates].copy()


def canonical_form(oracle: Oracle, f: FlatFsm):
    """Numbering-independent description of a DFA: (table, end bits, end-id tuples) in
    canonical BFS order.  Two DFAs are isomorphic iff these compare equal."""
    r = oracle.canonicalise(f)
    assert r is not None, "not a DFA"
    tab, cos = r
    n = tab.shape[0]
    inv = np.full(n, -1, dtype=np.int64)
    for s in range(f.nstates):
        if cos[s] != 0xFFFFFFFF:
            inv[cos[s]] = s
    ends = np.array([int(f.is_end[inv[c]]) for c in range(n)], dtype=np.uint8)
    ids = [tuple(int(x) for x in f.endids_of(int(inv[c]))) if ends[c] else () for c in range(n)]
    eager = [tuple(int(x) for x in f.eager_of(int(inv[c]))) for c in range(n)]
    return tab, ends, ids, eager


def canonical_digest(oracle, f):
    """sha256 over the numbering-independent form of a DFA (reflib.canonical_form): table, end bits, end-id sets."""
    import hashlib
    tab, ends, ids, _eager = canonical_form(oracle, f)
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(tab, dtype=np.uint32).tobytes())
    h.update(np.ascontiguousarray(ends, dtype=np.uint8).tobytes())
    for t in ids:
        h.update(np.asarray(t, dtype=np.uint32).tobytes() + b"|")
    return h.hexdigest()


class RefFlat(C.Structure):
    _fields_ = [("desc", CDesc), ("blocks", C.c_void_p * 8)]


class _Recipes:
    """Constructions built from the primitives, shared by Ref and RecordedRef."""

    def compile_dfa(self, pattern, dialect: int = RE_PCRE, flags: int = 0, minimise: bool = True,
                    endid: int | None = None):
        """re_comp -> fsm_determinise [-> fsm_minimise] [-> fsm_setendid]; returns handle."""
        h = self.re_comp(pattern, dialect, flags)
        self.determinise(h)
        if minimise:
            self.minimise(h)
        if endid is not None:
            self.setendid(h, endid)
        return h

    def union_dfa(self, patterns, dialect: int = RE_PCRE, flags: int = 0, minimise_each: bool = True,
                  state_limit: int = 0):
        """The rx(1)/re(1) recipe (reference src/rx/main.c:487-566,1353,1371): per pattern
        re_comp+determinise+minimise+setendid(index), fsm_union_array, fsm_determinise."""
        hs = [self.compile_dfa(p, dialect, flags, minimise_each, endid=i) for i, p in enumerate(patterns)]
        u = self.union_array(hs)
        if state_limit:
            res = self.determinise_limit(u, state_limit)
            if res != 0:
                self.free(u)
                raise RuntimeError(f"union determinise: result {res} (1 = state limit {state_limit} reached)")
        else:
            self.determinise(u)
        return u


class Ref(_Recipes):
    """The unmodified reference, through oracle/ref_harness.c."""

    def __init__(self):
        self.lib = C.CDLL(HARNESS_SO, use_errno=True)
        L, vp, P = self.lib, C.c_void_p, C.POINTER
        L.refh_re_comp.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_int]; L.refh_re_comp.restype = vp
        L.refh_parse_file.argtypes = [C.c_char_p]; L.refh_parse_file.restype = vp
        L.refh_determinise.argtypes = [vp]
        L.refh_determinise_limit.argtypes = [vp, C.c_size_t]
        L.refh_minimise.argtypes = [vp]
        L.refh_setendid.argtypes = [vp, C.c_uint]
        L.refh_union_array.argtypes = [C.c_size_t, P(vp)]; L.refh_union_array.restype = vp
        L.refh_clone.argtypes = [vp]; L.refh_clone.restype = vp
        L.refh_free.argtypes = [vp]; L.refh_free.restype = None
        L.refh_countstates.argtypes = [vp]; L.refh_countstates.restype = C.c_uint
        L.refh_equal.argtypes = [vp, vp]
        L.refh_remove_epsilons.argtypes = [vp]
        L.refh_from_desc.argtypes = [P(CDesc)]; L.refh_from_desc.restype = vp
        L.refh_flatten.argtypes = [vp, P(RefFlat)]
        L.refh_flat_free.argtypes = [P(RefFlat)]; L.refh_flat_free.restype = None
        L.refh_epsilon_closure.argtypes = [vp, P(vp), P(vp)]
        L.refh_exec.argtypes = [vp, vp, C.c_uint64, P(CResult)]
        L.refh_exec_batch.argtypes = [vp, vp, vp, C.c_size_t, C.c_int, C.c_int, vp]
        L.refh_endids.argtypes = [vp, C.c_uint, vp, C.c_size_t]; L.refh_endids.restype = C.c_size_t
        L.refh_eager_set.argtypes = [vp, C.c_uint, C.c_uint]
        L.refh_eager_flatten.argtypes = [vp, P(vp), P(vp)]
        L.refh_exec_eager.argtypes = [vp, vp, C.c_uint64, P(CResult), vp, C.c_size_t, P(C.c_size_t)]
        L.refh_union_repeated_pattern_group.argtypes = [C.c_size_t, P(vp), C.c_uint]
        L.refh_union_repeated_pattern_group.restype = vp
        L.refh_dfavm_bytes.argtypes = [vp, P(vp), P(C.c_size_t)]
        L.refh_vm_match_batch.argtypes = [vp, vp, vp, C.c_size_t, C.c_int, vp]
        L.refh_utf8dfa.argtypes = [C.c_int, C.c_int]; L.refh_utf8dfa.restype = vp
        L.refh_star.argtypes = [vp]
        L.refh_exec_eager_batch.argtypes = [vp, vp, vp, C.c_size_t, C.c_int, C.c_int, vp, vp, C.c_size_t, vp, C.c_size_t]
        self.libc = C.CDLL(None)
        self.libc.free.argtypes = [vp]

    # -- eager outputs ----------------------------------------------------------------
    def eager_set(self, h, state: int, ident: int) -> None:
        assert self.lib.refh_eager_set(h, state, ident) == 1

    def exec_eager(self, h, data: bytes):
        """(record, sorted fired ids) of one reference fsm_exec with the eager callback set."""
        buf = np.frombuffer(data, dtype=np.uint8)
        r = CResult()
        fired = np.zeros(256, dtype=np.uint32)
        n = C.c_size_t(0)
        self.lib.refh_exec_eager(h, _ptr(buf), len(data), C.byref(r), _ptr(fired), fired.size, C.byref(n))
        assert n.value <= fired.size
        return (r.ret, r.end, r.consumed), [int(x) for x in fired[:n.value]]

    def exec_eager_batch(self, h, base: np.ndarray, offsets: np.ndarray, id_of_bit: np.ndarray, mode: int = 1,
                         nthreads: int = 1):
        """(records, masks uint64 [n, words]) of n reference fsm_exec calls with the eager callback;
        bit b of a mask <=> id_of_bit[b] fired.  mode 0: fsm_exec as-is, mode 1: validation hoisted."""
        n = offsets.shape[0] - 1
        ids = np.ascontiguousarray(id_of_bit, dtype=np.uint32)
        words = max(1, (ids.size + 63) // 64)
        out = np.zeros(n, dtype=RESULT_DTYPE)
        masks = np.zeros((n, words), dtype=np.uint64)
        rc = self.lib.refh_exec_eager_batch(h, _ptr(base), offsets.ctypes.data, n, mode, nthreads, _ptr(out), _ptr(masks),
                                            words, _ptr(ids), ids.size)
        if rc != 0:
            raise OSError(C.get_errno(), "refh_exec_eager_batch")
        return out, masks

    def last_walk_seconds(self) -> float:
        """Seconds the worker threads of the last exec_eager_batch spent walking (excludes the per-thread fsm_clone)."""
        self.lib.refh_last_walk_seconds.restype = C.c_double
        return float(self.lib.refh_last_walk_seconds())

    def union_repeated_pattern_group(self, handles, id_base: int = 1):
        arr = (C.c_void_p * len(handles))(*handles)
        h = self.lib.refh_union_repeated_pattern_group(len(handles), arr, id_base)
        assert h
        return h

    # -- the DFAVM bytecode engine -----------------------------------------------------
    def dfavm_bytes(self, h) -> bytes:
        """The "DFAVM$" file image of a DFA: fsm_vm_compile + fsm_dfavm_save."""
        buf, n = C.c_void_p(), C.c_size_t(0)
        assert self.lib.refh_dfavm_bytes(h, C.byref(buf), C.byref(n)) == 0
        try:
            return C.string_at(buf, n.value)
        finally:
            self.libc.free(buf)

    def vm_match_batch(self, h, base: np.ndarray, offsets: np.ndarray, nthreads: int = 1) -> np.ndarray:
        n = offsets.shape[0] - 1
        out = np.zeros(n, dtype=np.uint8)
        assert self.lib.refh_vm_match_batch(h, _ptr(base), offsets.ctypes.data, n, nthreads, _ptr(out)) == 0
        return out

    # -- construction ---------------------------------------------------------------
    def utf8dfa(self, lo: int = 0, hi: int = 0x10FFFF):
        """examples/utf8dfa: the DFA that accepts exactly one UTF-8 encoded code point of lo..hi."""
        h = self.lib.refh_utf8dfa(lo, hi)
        assert h
        return h

    def star(self, h) -> None:
        assert self.lib.refh_star(h) == 1

    def re_comp(self, pattern: str | bytes, dialect: int = RE_PCRE, flags: int = 0):
        p = pattern.encode() if isinstance(pattern, str) else pattern
        h = self.lib.refh_re_comp(p, len(p), dialect, flags)
        if not h:
            raise ValueError(f"re_comp failed for {pattern!r}")
        return h

    def parse_file(self, path: str):
        h = self.lib.refh_parse_file(path.encode())
        if not h:
            raise ValueError(f"fsm_parse failed for {path}")
        return h

    def determinise(self, h) -> None:
        assert self.lib.refh_determinise(h) == 1

    def determinise_limit(self, h, limit: int) -> int:
        return int(self.lib.refh_determinise_limit(h, limit))

    def minimise(self, h) -> None:
        assert self.lib.refh_minimise(h) == 1

    def setendid(self, h, i: int) -> None:
        assert self.lib.refh_setendid(h, i) == 1

    def union_array(self, handles):
        arr = (C.c_void_p * len(handles))(*handles)
        h = self.lib.refh_union_array(len(handles), arr)
        assert h
        return h

    def clone(self, h):
        return self.lib.refh_clone(h)

    def free(self, h) -> None:
        self.lib.refh_free(h)

    def countstates(self, h) -> int:
        return int(self.lib.refh_countstates(h))

    def equal(self, a, b) -> bool:
        return self.lib.refh_equal(a, b) == 1

    def remove_epsilons(self, h) -> None:
        assert self.lib.refh_remove_epsilons(h) == 1

    def from_flat(self, f: FlatFsm):
        d = f.as_c()
        h = self.lib.refh_from_desc(C.byref(d))
        assert h
        return h

    def flatten(self, h) -> FlatFsm:
        rf = RefFlat()
        assert self.lib.refh_flatten(h, C.byref(rf)) == 0
        try:
            f = FlatFsm.from_c(rf.desc)
        finally:
            self.lib.refh_flat_free(C.byref(rf))
        off, ids = C.c_void_p(), C.c_void_p()
        assert self.lib.refh_eager_flatten(h, C.byref(off), C.byref(ids)) == 0
        try:
            eo = np.ctypeslib.as_array(C.cast(off, C.POINTER(C.c_uint64)), shape=(f.nstates + 1,)).copy()
            if int(eo[-1]) > 0:
                f.eager_off = eo
                f.eager_ids = np.ctypeslib.as_array(C.cast(ids, C.POINTER(C.c_uint32)), shape=(int(eo[-1]),)).copy()
        finally:
            self.libc.free(off); self.libc.free(ids)
        return f

    # -- execution --------------------------------------------------------------------
    def epsilon_closure(self, h, nstates: int):
        off, to = C.c_void_p(), C.c_void_p()
        assert self.lib.refh_epsilon_closure(h, C.byref(off), C.byref(to)) == 0
        o = np.frombuffer((C.c_uint64 * (nstates + 1)).from_address(off.value), dtype=np.uint64).copy()
        t = np.frombuffer((C.c_uint32 * max(int(o[-1]), 1)).from_address(to.value), dtype=np.uint32)[:int(o[-1])].copy()
        self.libc.free(off); self.libc.free(to)
        return o, t

    def exec(self, h, data: bytes):
        buf = np.frombuffer(data, dtype=np.uint8) if len(data) else np.zeros(0, np.uint8)
        r = CResult()
        rc = self.lib.refh_exec(h, _ptr(buf), len(data), C.byref(r))
        return rc, int(r.end), int(r.consumed)

    def exec_batch(self, h, base: np.ndarray, offsets: np.ndarray, mode: int = 1, nthreads: int = 1) -> np.ndarray:
        n = offsets.shape[0] - 1
        out = np.zeros(n, dtype=RESULT_DTYPE)
        rc = self.lib.refh_exec_batch(h, _ptr(base), offsets.ctypes.data, n, mode, nthreads, _ptr(out))
        if rc != 0:
            raise OSError(C.get_errno(), "refh_exec_batch")
        return out

    def exec_batch_digest(self, h, base: np.ndarray, offsets: np.ndarray, mode: int = 1, nthreads: int = 1) -> str:
        """records_digest of exec_batch: the answer for batches too large to record."""
        return records_digest(self.exec_batch(h, base, offsets, mode=mode, nthreads=nthreads))

    def exec_eager_batch_digest(self, h, base: np.ndarray, offsets: np.ndarray, id_of_bit: np.ndarray, mode: int = 1,
                                nthreads: int = 1) -> str:
        """records_digest of exec_eager_batch (records and id bitsets)."""
        return records_digest(*self.exec_eager_batch(h, base, offsets, id_of_bit, mode=mode, nthreads=nthreads))

    def numbering(self, h) -> str:
        """numbering_digest of the automaton as it stands: its states, numbered as the reference numbers them."""
        f = self.flatten(h)
        return numbering_digest(f.dense_table(), f.is_end)

    def endids(self, h, state: int):
        buf = (C.c_uint * 4096)()
        c = self.lib.refh_endids(h, state, buf, 4096)
        return [int(buf[i]) for i in range(min(c, 4096))]


# -- the reference's answers, recorded -----------------------------------------------------------
#
# Tests that compare with the reference get it from reference(): the compiled harness where it was
# built, otherwise RecordedRef, which answers every query the suite makes from REF_CALLS, a record
# of the harness's own answers.  An automaton is named by a hash of the calls that built it (inputs
# included), a query by that name plus its arguments.  Batches of hundreds of thousands of records are
# asked for as a digest (records_digest).  FSM_B200_REF=record runs the live harness and writes its
# answers to REF_CALLS; FSM_B200_REF=replay uses the record even where the harness exists.

REF_CALLS = os.path.join(ROOT, "tests", "golden", "ref_calls.json.xz")
REF_MODE = os.environ.get("FSM_B200_REF", "")


def replaying() -> bool:
    """True when reference() answers from REF_CALLS rather than from the compiled harness."""
    return REF_MODE == "replay" or (REF_MODE != "record" and not have_ref())


def reference():
    if REF_MODE == "record":
        return RecordedRef(live=Ref())
    return RecordedRef() if replaying() else Ref()


def _key(*parts) -> str:
    m = hashlib.sha256()
    for p in parts:
        if isinstance(p, FlatFsm):
            p = (p.nstates, p.start, bool(p.hasstart), p.is_end, p.group_off, p.group_symbols, p.group_to, p.eps_off,
                 p.eps_to, p.endid_off, p.endids, p.eager_off, p.eager_ids)
        if isinstance(p, (np.integer, np.bool_)):
            p = p.item()                             # numpy scalars key like the Python value they hold
        if isinstance(p, tuple):
            m.update(_key(*p).encode())
        elif isinstance(p, np.ndarray):
            m.update(f"{p.dtype.str}{p.shape}".encode() + np.ascontiguousarray(p).tobytes())
        else:
            m.update(repr(p).encode() if not isinstance(p, bytes) else p)
        m.update(b"\0")
    return m.hexdigest()[:32]


def records_digest(records: np.ndarray, masks: np.ndarray | None = None) -> str:
    """Digest of result records (and of the eager-output id bitsets [n, words] that go with them)."""
    r = np.ascontiguousarray(records, dtype=RESULT_DTYPE)
    if masks is None:
        return _key(r)
    return _key(r, np.ascontiguousarray(masks, dtype=np.uint64).reshape(r.shape[0], -1))


def numbering_digest(table: np.ndarray, is_end: np.ndarray) -> str:
    """Digest of a DFA's dense transition table [nstates, 256] and end bits, state numbering included."""
    return _key(np.ascontiguousarray(table, dtype=np.uint32), np.asarray(is_end).astype(bool))


def _to_json(v):
    if isinstance(v, FlatFsm):
        return {"fsm": [v.nstates, v.start, bool(v.hasstart)] +
                       [None if a is None else a.reshape(-1).tolist() for a in
                        (v.is_end, v.group_off, v.group_symbols, v.group_to, v.eps_off, v.eps_to, v.endid_off,
                         v.endids, v.eager_off, v.eager_ids)]}
    if isinstance(v, np.ndarray):
        fields = v.dtype.names or (None,)
        return {"nd": np.lib.format.dtype_to_descr(v.dtype), "shape": list(v.shape),
                "v": [(v[f] if f else v).reshape(-1).tolist() for f in fields]}
    if isinstance(v, bytes):
        return {"bytes": base64.b64encode(v).decode()}
    if isinstance(v, tuple):
        return {"tuple": [_to_json(x) for x in v]}
    if isinstance(v, list):
        return [_to_json(x) for x in v]
    if isinstance(v, (np.integer, np.bool_)):
        return v.item()
    assert v is None or isinstance(v, (int, bool, str)), type(v)
    return v


def _from_json(j):
    if isinstance(j, list):
        return [_from_json(x) for x in j]
    if not isinstance(j, dict):
        return j
    if "fsm" in j:
        n, start, hasstart, *a = j["fsm"]
        return FlatFsm(n, start, hasstart, np.array(a[0], np.uint8), np.array(a[1], np.uint64),
                       np.array(a[2], np.uint64).reshape(-1, 4), np.array(a[3], np.uint32), np.array(a[4], np.uint64),
                       np.array(a[5], np.uint32), np.array(a[6], np.uint64), np.array(a[7], np.uint32),
                       None if a[8] is None else np.array(a[8], np.uint64), None if a[9] is None else np.array(a[9], np.uint32))
    if "nd" in j:
        dt = np.lib.format.descr_to_dtype(j["nd"] if isinstance(j["nd"], str) else [tuple(d) for d in j["nd"]])
        out = np.empty(j["shape"], dtype=dt)
        for f, v in zip(dt.names or (None,), j["v"]):
            (out[f] if f else out).reshape(-1)[:] = v
        return out
    if "bytes" in j:
        return base64.b64decode(j["bytes"])
    return tuple(_from_json(x) for x in j["tuple"])


class _Handle:
    """An automaton of RecordedRef: the hash of the calls that built it (and the live handle when recording)."""

    def __init__(self, key: str, live=None):
        self.key, self.live = key, live


class RecordedRef(_Recipes):
    """Ref's interface over REF_CALLS; with `live`, the compiled harness answers and REF_CALLS records it.
    A record is made from scratch by one run of the whole suite (GPU tests included), so that it holds
    exactly the calls the suite makes."""
    _saved: dict | None = None

    def __init__(self, live: Ref | None = None):
        self.live = live
        if RecordedRef._saved is None:
            RecordedRef._saved = {}
            if live is not None:
                atexit.register(RecordedRef._write)
            elif os.path.exists(REF_CALLS):
                with lzma.open(REF_CALLS, "rt") as fh:
                    RecordedRef._saved = json.load(fh)
        self.calls = RecordedRef._saved

    @staticmethod
    def _write():
        with lzma.open(REF_CALLS, "wt", preset=9 | lzma.PRESET_EXTREME) as fh:
            json.dump(RecordedRef._saved, fh, separators=(",", ":"), sort_keys=True)

    def _answer(self, key: str, ask):
        if self.live is not None:
            v = ask()
            self.calls[key] = _to_json(v)
            return v
        if key not in self.calls:
            raise LookupError(f"no recorded answer of the reference for this call ({key}); "
                              f"record it with FSM_B200_REF=record where the compiled reference is built")
        return _from_json(self.calls[key])

    def _new(self, key: str, make) -> _Handle:
        return _Handle(key, make() if self.live is not None else None)

    def _mutate(self, h: _Handle, op: str, *args) -> None:
        if self.live is not None:
            getattr(self.live, op)(h.live, *args)
        h.key = _key(op, h.key, *args)

    # -- construction
    def parse_file(self, path: str):
        raise NotImplementedError("parse_file reads a file of the reference's tree: it needs the compiled reference")

    def re_comp(self, pattern, dialect: int = RE_PCRE, flags: int = 0):
        p = pattern.encode() if isinstance(pattern, str) else pattern
        key = _key("re_comp", p, dialect, flags)
        live = []

        def ask():
            try:
                live.append(self.live.re_comp(p, dialect, flags))
                return True
            except ValueError:
                return False
        if not self._answer(key, ask):
            raise ValueError(f"re_comp failed for {pattern!r}")
        return _Handle(key, live[0] if live else None)

    def from_flat(self, f: FlatFsm):
        return self._new(_key("from_flat", f), lambda: self.live.from_flat(f))

    def utf8dfa(self, lo: int = 0, hi: int = 0x10FFFF):
        return self._new(_key("utf8dfa", lo, hi), lambda: self.live.utf8dfa(lo, hi))

    def union_array(self, handles):
        return self._new(_key("union_array", *[h.key for h in handles]),
                         lambda: self.live.union_array([h.live for h in handles]))

    def union_repeated_pattern_group(self, handles, id_base: int = 1):
        return self._new(_key("union_repeated_pattern_group", id_base, *[h.key for h in handles]),
                         lambda: self.live.union_repeated_pattern_group([h.live for h in handles], id_base))

    def clone(self, h):
        return self._new(h.key, lambda: self.live.clone(h.live))

    def free(self, h) -> None:
        if self.live is not None:
            self.live.free(h.live)

    # -- in-place operations
    def determinise(self, h) -> None:
        self._mutate(h, "determinise")

    def minimise(self, h) -> None:
        self._mutate(h, "minimise")

    def setendid(self, h, i: int) -> None:
        self._mutate(h, "setendid", i)

    def remove_epsilons(self, h) -> None:
        self._mutate(h, "remove_epsilons")

    def star(self, h) -> None:
        self._mutate(h, "star")

    def eager_set(self, h, state: int, ident: int) -> None:
        self._mutate(h, "eager_set", state, ident)

    def determinise_limit(self, h, limit: int) -> int:
        r = self._answer(_key("determinise_limit", h.key, limit), lambda: self.live.determinise_limit(h.live, limit))
        h.key = _key("determinise_limit", h.key, limit)
        return r

    # -- queries
    def flatten(self, h) -> FlatFsm:
        return self._answer(_key("flatten", h.key), lambda: self.live.flatten(h.live))

    def numbering(self, h) -> str:
        return self._answer(_key("numbering", h.key), lambda: self.live.numbering(h.live))

    def countstates(self, h) -> int:
        return self._answer(_key("countstates", h.key), lambda: self.live.countstates(h.live))

    def equal(self, a, b) -> bool:
        return self._answer(_key("equal", a.key, b.key), lambda: self.live.equal(a.live, b.live))

    def endids(self, h, state: int):
        return self._answer(_key("endids", h.key, state), lambda: self.live.endids(h.live, state))

    def exec(self, h, data: bytes):
        return self._answer(_key("exec", h.key, bytes(data)), lambda: self.live.exec(h.live, data))

    def exec_eager(self, h, data: bytes):
        return self._answer(_key("exec_eager", h.key, bytes(data)), lambda: self.live.exec_eager(h.live, data))

    def exec_batch(self, h, base: np.ndarray, offsets: np.ndarray, mode: int = 1, nthreads: int = 1) -> np.ndarray:
        return self._answer(_key("exec_batch", h.key, base, offsets, mode),
                            lambda: self.live.exec_batch(h.live, base, offsets, mode=mode, nthreads=nthreads))

    def exec_batch_digest(self, h, base: np.ndarray, offsets: np.ndarray, mode: int = 1, nthreads: int = 1) -> str:
        return self._answer(_key("exec_batch_digest", h.key, base, offsets, mode),
                            lambda: self.live.exec_batch_digest(h.live, base, offsets, mode=mode, nthreads=nthreads))

    def exec_eager_batch_digest(self, h, base: np.ndarray, offsets: np.ndarray, id_of_bit: np.ndarray, mode: int = 1,
                                nthreads: int = 1) -> str:
        return self._answer(_key("exec_eager_batch_digest", h.key, base, offsets, np.asarray(id_of_bit), mode),
                            lambda: self.live.exec_eager_batch_digest(h.live, base, offsets, id_of_bit, mode=mode,
                                                                      nthreads=nthreads))

    def exec_eager_batch(self, h, base: np.ndarray, offsets: np.ndarray, id_of_bit: np.ndarray, mode: int = 1,
                         nthreads: int = 1):
        return self._answer(_key("exec_eager_batch", h.key, base, offsets, np.asarray(id_of_bit), mode),
                            lambda: self.live.exec_eager_batch(h.live, base, offsets, id_of_bit, mode=mode, nthreads=nthreads))

    def epsilon_closure(self, h, nstates: int):
        return self._answer(_key("epsilon_closure", h.key, nstates), lambda: self.live.epsilon_closure(h.live, nstates))

    def dfavm_bytes(self, h) -> bytes:
        return self._answer(_key("dfavm_bytes", h.key), lambda: self.live.dfavm_bytes(h.live))

    def vm_match_batch(self, h, base: np.ndarray, offsets: np.ndarray, nthreads: int = 1) -> np.ndarray:
        return self._answer(_key("vm_match_batch", h.key, base, offsets),
                            lambda: self.live.vm_match_batch(h.live, base, offsets, nthreads=nthreads))
