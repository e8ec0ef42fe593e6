"""GPU: the drop-in boundary.  The reference's re(1) relinked, UNCHANGED, against the shim
(reference libfsm minus src/libfsm/exec.c plus libfsm_b200/shim/fsm_b200_shim.c): same exit
status and output as the reference's own re(1) -- BASELINE config 1's plumbing."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RE_B200 = os.path.join(ROOT, "build", "shim", "re_b200")
RE_REF = os.path.join(ROOT, "oracle", "_ref", "re_ref")

needs_bins = pytest.mark.skipif(not (os.path.exists(RE_B200) and os.path.exists(RE_REF)),
                                reason="relinked CLIs not built (need the reference tree at build time)")


def run(binary, args):
    p = subprocess.run([binary] + args, capture_output=True, timeout=120)
    return p.returncode, p.stdout, p.stderr


@needs_bins
def test_config1_files(tmp_path):
    """re -r pcre -x '[0-9]+\\.[0-9]+' FILE over 1 MiB of seeded ASCII (SURVEY.md 8d config 1)."""
    rng = np.random.default_rng(1)
    match = rng.integers(ord("0"), ord("9") + 1, size=1 << 20, dtype=np.uint8)
    match[rng.random(match.size) < 1 / 64] = ord(".")
    nomatch = rng.integers(ord("a"), ord("z") + 1, size=1 << 20, dtype=np.uint8)
    fm, fn = tmp_path / "match.txt", tmp_path / "nomatch.txt"
    fm.write_bytes(match.tobytes()); fn.write_bytes(nomatch.tobytes())
    for files in ([str(fm)], [str(fn)], [str(fm), str(fn)], [str(fn), str(fm)]):
        args = ["-r", "pcre", "-x", r"[0-9]+\.[0-9]+"] + files
        got, want = run(RE_B200, args), run(RE_REF, args)
        assert got[0] == want[0] and got[1] == want[1], (files, got, want)
    assert run(RE_B200, ["-r", "pcre", "-x", r"[0-9]+\.[0-9]+", str(fm)])[0] == 0
    assert run(RE_B200, ["-r", "pcre", "-x", r"[0-9]+\.[0-9]+", str(fn)])[0] == 1


@needs_bins
def test_re_x_large_file_against_the_reference(tmp_path):
    """`re -x PATTERN FILE` on a 512 MiB file that has to be read to its end (whole-file pattern): the
    relinked, unchanged re(1) -- fsm_fgetc recognised by the shim and read in fread blocks, K1b over the
    buffer -- gives the reference's verdict, in less than the reference's time (one fgetc + one group
    scan per byte).  The timings are printed."""
    import time
    rng = np.random.default_rng(3)
    n = 512 << 20
    data = rng.integers(ord("a"), ord("z") + 1, size=n, dtype=np.uint8)
    data[rng.random(n, dtype=np.float32) < 0.15] = ord(" ")
    good, bad = tmp_path / "good.txt", tmp_path / "bad.txt"
    good.write_bytes(data.tobytes())
    data[n - 12345] = ord("#")
    bad.write_bytes(data.tobytes())
    del data
    times = {}
    for name, f, want_rc in (("good", good, 0), ("bad", bad, 1)):
        args = ["-r", "pcre", "-x", r"^[a-z ]+$", str(f)]
        t0 = time.perf_counter(); got = run(RE_B200, args); t1 = time.perf_counter(); want = run(RE_REF, args); t2 = time.perf_counter()
        assert got[0] == want[0] == want_rc and got[1] == want[1], (name, got, want)
        times[name] = {"re_b200_s": t1 - t0, "re_ref_s": t2 - t1}
    print("re -x 512 MiB:", times)
    assert times["good"]["re_b200_s"] < times["good"]["re_ref_s"], times


@needs_bins
@pytest.mark.parametrize("args", [
    ["-r", "pcre", r"a[ -~]{7}\z", "xxabcdefgh"],
    ["-r", "pcre", r"a[ -~]{7}\z", "xxabcdefg"],
    ["-r", "pcre", r"^abc[0-9]+x$", "abc123x", "abc12", "zzz"],
    ["-r", "native", "ab*c", "abbbc"],
    ["-r", "glob", "*.txt", "notes.txt"],
    ["-r", "literal", "hello", "hello"],
])
def test_argv_strings_same_exit_status(args):
    got, want = run(RE_B200, args), run(RE_REF, args)
    assert got[0] == want[0] and got[1] == want[1], (args, got, want)


@needs_bins
def test_multi_pattern_prints_matching_pattern():
    """re -z: several patterns (end id = argv index), `match: /pattern/` printed from the end id."""
    args = ["-r", "pcre", "-z", "-y", "/dev/null"]
    # patterns come from -y FILE or -s; use the simplest form both binaries accept
    args = ["-r", "pcre", "-z", "abc", "def", "xyz"]
    got, want = run(RE_B200, args), run(RE_REF, args)
    assert got[0] == want[0] and got[1] == want[1]


FSM_B200 = os.path.join(ROOT, "build", "shim", "fsm_b200")
FSM_REF = os.path.join(ROOT, "oracle", "_ref", "fsm_ref")


def to_fsm5(f) -> str | None:
    """A FlatFsm as fsm(5) text (printable labels only; None if it has others)."""
    lines = []
    for s in range(f.nstates):
        for g in range(int(f.group_off[s]), int(f.group_off[s + 1])):
            for c in range(256):
                if (int(f.group_symbols[g][c >> 6]) >> (c & 63)) & 1:
                    if not (0x20 <= c < 0x7F) or chr(c) in "'\\":
                        return None
                    lines.append(f"{s} -> {int(f.group_to[g])} '{chr(c)}';")
        for e in range(int(f.eps_off[s]), int(f.eps_off[s + 1])):
            lines.append(f"{s} -> {int(f.eps_to[e])};")
    if f.hasstart:
        lines.append(f"start: {f.start};")
    ends = [str(s) for s in range(f.nstates) if f.is_end[s]]
    if ends:
        lines.append("end: " + ", ".join(ends) + ";")
    return "\n".join(lines) + "\n"


@pytest.mark.skipif(not (os.path.exists(FSM_B200) and os.path.exists(FSM_REF)), reason="relinked fsm(1) not built")
def test_fsm_cli_determinise_like_the_reference_tests(tmp_path):
    """The reference's own test method for determinise (tests/determinise/Makefile:11-20):
    `fsm -pd in.fsm` then `fsm -t equal` against the expected automaton -- here with the
    relinked fsm(1) (fsm_determinise -> K2 on the GPU) against the reference's fsm(1)."""
    import goldenio
    cases = goldenio.load_det_cases(os.path.join(goldenio.GOLDEN_DIR, "golden_determinise.npz"))
    ran = 0
    for c in cases:
        if not (c["name"].startswith("determinise:") or c["name"].startswith("eclosure:") or c["name"] == "cfg5:20x6"):
            continue
        txt = to_fsm5(c["nfa"])
        if txt is None:
            continue
        inp = tmp_path / "in.fsm"
        inp.write_text(txt)
        outs = {}
        for tag, binary in (("b200", FSM_B200), ("ref", FSM_REF)):
            p = subprocess.run([binary, "-pd"], stdin=open(inp), capture_output=True, timeout=120)
            assert p.returncode == 0, (c["name"], tag, p.stderr)
            outs[tag] = tmp_path / f"out_{tag}.fsm"
            outs[tag].write_bytes(p.stdout)
        eq = subprocess.run([FSM_REF, "-t", "equal", str(outs["b200"]), str(outs["ref"])], capture_output=True, timeout=120)
        assert eq.returncode == 0, (c["name"], eq.stdout, eq.stderr)
        # same number of states too (subset construction without minimisation is canonical)
        cnt = [subprocess.run([FSM_REF, "-q", "count"], stdin=open(outs[t]), capture_output=True).stdout for t in ("b200", "ref")]
        assert cnt[0] == cnt[1], c["name"]
        ran += 1
    assert ran >= 10


SELFTEST = os.path.join(ROOT, "build", "shim", "shim_selftest")


@pytest.mark.skipif(not os.path.exists(SELFTEST), reason="shim selftest not built")
def test_shim_selftest_c_program():
    """A C program using only libfsm's API (re_comp, fsm_determinise, fsm_minimise,
    fsm_union_array, fsm_exec, fsm_endid_get) plus the additive fsm_exec_batch, linked to the
    shim: determinise runs through K2, exec through K1/K1b; see libfsm_b200/shim/shim_selftest.c."""
    p = subprocess.run([SELFTEST], capture_output=True, timeout=300)
    assert p.returncode == 0, (p.stdout.decode(), p.stderr.decode())
    assert b"shim selftest ok" in p.stdout


REFTESTS_DIR = os.path.join(ROOT, "build", "shim", "reftests")
# tests/eager_output/*.c run from tests/test_gpu_eager.py
REFTESTS = sorted(x for x in os.listdir(REFTESTS_DIR) if not x.startswith("eager_output")) if os.path.isdir(REFTESTS_DIR) else []


@pytest.mark.skipif(not REFTESTS, reason="reference unit tests not built against the shim")
@pytest.mark.parametrize("name", REFTESTS)
def test_reference_own_c_unit_tests_pass_against_the_shim(name):
    """The reference's own C unit tests (tests/endids/*.c, tests/re_strings/*.c), compiled
    unmodified from the reference tree and linked to the shim, so their fsm_determinise /
    fsm_minimise / fsm_exec calls run on the GPU; they assert internally and exit 0."""
    p = subprocess.run([os.path.join(REFTESTS_DIR, name)], capture_output=True, timeout=300)
    assert p.returncode == 0, (name, p.stdout.decode()[-2000:], p.stderr.decode()[-2000:])


FIXTURES_NPZ = os.path.join(ROOT, "tests", "golden", "golden_re_fixtures.npz")


def _fixtures():
    import goldenio
    return goldenio.load_re_fixtures(FIXTURES_NPZ) if os.path.exists(FIXTURES_NPZ) else []


@needs_bins
def test_reference_regex_golden_files_through_re_b200(ref, tmp_path):
    """The reference's regex golden-file tests (tests/pcre, pcre-anchor, pcre-repeat, pcre-flags,
    native, glob, like, literal, sql: `re -r D -py inN.re` compared with outN.fsm by language
    equality, tests/pcre/Makefile:44-78) replayed with the relinked re(1): re_comp is the
    reference's, fsm_determinise / fsm_minimise run through K2 / K3, the comparator is the
    reference's fsm_equal."""
    fixtures = _fixtures()
    assert len(fixtures) >= 200
    if not os.environ.get("FSM_B200_ALL_FIXTURES"):
        fixtures = fixtures[::10]         # each re(1) run is a fresh process (CUDA start-up + 5 engine calls ~1.7 s); all 267 pass with FSM_B200_ALL_FIXTURES=1
    bad = []
    for k, fx in enumerate(fixtures):
        rf = tmp_path / "in.re"
        rf.write_bytes(fx["regex"])
        p = subprocess.run([RE_B200] + fx["args"] + ["-r", fx["dialect"], "-py", str(rf)], capture_output=True, timeout=120)
        if p.returncode != 0:
            bad.append((fx["name"], "exit", p.returncode, p.stderr[-200:]))
            continue
        gf = tmp_path / "got.fsm"
        gf.write_bytes(p.stdout)
        hg = ref.parse_file(str(gf))
        he = ref.from_flat(fx["fsm"])
        if not ref.equal(hg, he):
            bad.append((fx["name"], "language differs"))
        ref.free(hg); ref.free(he)
    assert not bad, bad[:10]
