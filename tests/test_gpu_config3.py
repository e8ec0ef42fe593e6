"""GPU: BASELINE config 3 shape -- an rx(1)-style many-pattern union DFA (built by the reference:
per pattern re_comp/determinise/minimise/setendid, fsm_union_array, determinise; reference
src/rx/main.c:487-566,1353,1371) over ragged log lines.  Every record AND the end-id set of every
match are compared with the reference's own fsm_exec walk (live, or its recorded answers: for
batches of hundreds of thousands of lines, a digest of all records and id bitsets)."""
import numpy as np
import pytest

import reflib
import libfsm_b200 as L

pytestmark = [pytest.mark.gpu]


def build_patterns(npat, rng):
    words = ["ERROR", "WARN", "INFO", "DEBUG", "FATAL", "kernel", "sshd", "nginx", "cron", "systemd"]
    templates = [lambda w, k: (f"^{w} [0-9]{{{k}}} ", f"{w} {'7' * k} "),
                 lambda w, k: (f"^{w}: user=[a-z]+ id=[0-9]{{{k}}}", f"{w}: user=bob id={'4' * k}"),
                 lambda w, k: (f"^{w}\\[[0-9]+\\]: ", f"{w}[123]: "),
                 lambda w, k: (f"^{w} (GET|POST|PUT) /[a-z/]+ ", f"{w} GET /a/b "),
                 lambda w, k: (f"^{w} [A-Z]{{{k}}}-[0-9]+", f"{w} {'Q' * k}-99")]
    pats, exs = [], []
    while len(pats) < npat:
        w = words[int(rng.integers(len(words)))] + str(int(rng.integers(0, 30)))
        p, e = templates[int(rng.integers(len(templates)))](w, int(rng.integers(1, 4)))
        if p not in pats:
            pats.append(p); exs.append(e.encode())
    return pats, exs


@pytest.mark.parametrize("npat", [24, 96])
def test_union_dfa_over_ragged_lines(ref, oracle, npat):
    rng = np.random.default_rng(7 + npat)
    pats, exs = build_patterns(npat, rng)
    h = ref.union_dfa(pats, state_limit=200000)
    fsm = ref.flatten(h)
    nlines = 300000
    lens = rng.integers(0, 257, size=nlines)
    lines = []
    noise = rng.integers(0x20, 0x7F, size=int(lens.sum()) + 64, dtype=np.uint8)
    pos = 0
    for i in range(nlines):
        body = noise[pos:pos + int(lens[i])].tobytes(); pos += int(lens[i])
        if i % 2 == 0:
            e = exs[int(rng.integers(len(exs)))]
            body = (e + body)[:max(len(body), 0)] if i % 4 == 0 else e[:len(e) // 2] + body
        lines.append(body)
    base, off = reflib.offsets_for(lines)
    # the reference's own walk, through the oracle's records pinned to it by digest (the oracle's show
    # which line differs); then fsm_endid_get of every end state the first 500 matches reach
    want = oracle.exec_batch(fsm, base, off, nthreads=16)
    assert reflib.records_digest(want) == ref.exec_batch_digest(h, base, off, mode=1, nthreads=16)
    assert 0.05 < (want["ret"] == 1).mean() < 0.9
    matched = np.nonzero(want["ret"] == 1)[0][:500]
    want_ids = {s: ref.endids(h, s) for s in sorted({int(want["end"][i]) for i in matched})}
    ref.free(h)
    with L.Dfa(fsm) as dfa:
        got = dfa.exec_batch(base, off)                            # host path -> ragged kernel
        import torch
        dout = dfa.exec_batch(torch.from_numpy(base).cuda(), torch.from_numpy(off.astype(np.int64)).cuda())
        torch.cuda.synchronize()
        assert dfa.info["entry_bytes"] == 2 or fsm.nstates <= 255
    assert (got == want).all()
    assert (L.results_from_torch(dout) == want).all()
    # end ids through the flat description == fsm_endid_get of the reference
    for i in matched:
        assert list(fsm.endids_of(int(got["end"][i]))) == want_ids[int(want["end"][i])]


# ---- the two config-3 automata of tests/golden/golden_cfg3.npz (built by the reference) ---------

@pytest.fixture(scope="module")
def cfg3():
    import goldenio
    return goldenio.load_cfg3()


def test_cfg3_eager_golden_lines(cfg3):
    """128 mostly unanchored patterns, fsm_union_repeated_pattern_group + det + min: records and fired
    eager-output id sets of the golden sample, through the host entry point and through the device
    entry point (lines kernel), bit-exact vs what the reference's fsm_exec + callback produced."""
    import torch
    c = cfg3["eager"]
    with L.Dfa(c["fsm"]) as dfa:
        assert dfa.info["lines_smem"] == 1 and dfa.info["eager_ids"] == c["idlist"].size
        assert (dfa.eager_ids() == c["idlist"]).all()
        rec, masks = dfa.exec_batch_eager(c["base"], c["offsets"])
        assert (rec == c["expect"]).all()
        assert (masks == c["masks"]).all()
        drec, dmasks = dfa.exec_batch_eager(torch.from_numpy(c["base"]).cuda(), torch.from_numpy(c["offsets"].astype(np.int64)).cuda())
        torch.cuda.synchronize()
        assert (L.results_from_torch(drec) == c["expect"]).all()
        assert (dmasks.cpu().numpy().view(np.uint64) == c["masks"]).all()
        # the plain entry points on the same automaton: same records, no ids
        assert (dfa.exec_batch(c["base"], c["offsets"]) == c["expect"]).all()
    assert (c["masks"] != 0).any(axis=1).mean() > 0.3 and (c["expect"]["ret"] == 1).any()


def test_cfg3_anchored_golden_lines(cfg3):
    c = cfg3["anchored"]
    with L.Dfa(c["fsm"]) as dfa:
        assert dfa.info["lines_smem"] == 1
        assert (dfa.exec_batch(c["base"], c["offsets"]) == c["expect"]).all()
    assert 0.2 < (c["expect"]["ret"] == 1).mean() < 0.8


@pytest.mark.parametrize("lo,hi", [(0, 40), (64, 256), (1, 1000)])
def test_cfg3_eager_vs_reference_large_sample(ref, cfg3, lo, hi):
    """300 k seeded lines (incl. empty lines and lines much longer than a sector) through the lines
    kernel vs the compiled reference (refh_exec_eager_batch: its own edge_set_transition walk and
    fsm_eager_output_iter_state per state entered), records + id bitsets bit-exact; and the absorbing
    exit / NOP-column machinery at every alignment (the lines are packed back to back)."""
    import torch
    from libfsm_b200 import workloads
    c = cfg3["eager"]
    _, inst = workloads.cfg3_patterns()
    base, off = workloads.cfg3_lines_host(300000 if hi <= 256 else 60000, inst, seed=lo * 7 + hi, lo=lo, hi=hi)
    h = ref.from_flat(c["fsm"])
    want = ref.exec_eager_batch_digest(h, base, off, c["idlist"], mode=1, nthreads=16)
    ref.free(h)
    with L.Dfa(c["fsm"]) as dfa:
        drec, dmasks = dfa.exec_batch_eager(torch.from_numpy(base).cuda(), torch.from_numpy(off.astype(np.int64)).cuda())
        torch.cuda.synchronize()
        got, gmasks = L.results_from_torch(drec), dmasks.cpu().numpy().view(np.uint64)
    assert reflib.records_digest(got, gmasks) == want, "records or id bitsets differ from the reference's"


def test_cfg3_eager_host_path_pipelines_chunks(ref, cfg3, monkeypatch):
    """fsm_b200_exec_batch_eager_host cuts a batch into chunks that alternate between two slots (copy-in of
    one overlaps scan + copy-out of the other): with 1 MiB chunks a 100 k-line batch takes dozens of them,
    at every alignment; records and id bitsets must equal the reference's, line for line."""
    from libfsm_b200 import workloads
    c = cfg3["eager"]
    _, inst = workloads.cfg3_patterns()
    base, off = workloads.cfg3_lines_host(100000, inst, seed=99, lo=0, hi=300)
    h = ref.from_flat(c["fsm"])
    want = ref.exec_eager_batch_digest(h, base, off, c["idlist"], mode=1, nthreads=16)
    ref.free(h)
    monkeypatch.setenv("FSM_B200_HOST_CHUNK_MB", "1")
    with L.Dfa(c["fsm"]) as dfa:
        L.launch_count(reset=True)
        rec, masks = dfa.exec_batch_eager(base, off)
        assert L.launch_count() >= 10
        assert reflib.records_digest(rec, masks) == want, "records or id bitsets differ from the reference's"
        # a sub-range that does not start at offset 0: the same lines' records (equal to the reference's above)
        rec2, masks2 = dfa.exec_batch_eager(base, off[5000:60001])
        assert (rec2 == rec[5000:60000]).all() and (masks2 == masks[5000:60000]).all()
