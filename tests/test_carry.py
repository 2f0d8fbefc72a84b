"""Carry coverage of the device arithmetic, on the CPU.  The carry corpus (tests/carry_corpus.py) runs through the simulation of
the device code built with the carry sanitizer (tests/hostsim/carry_trace.cpp, build_carry.sh), which sees every carry primitive
of arith.cuh with its call site.  Checked:
  - every row equals its reference (the C oracle where it has the op, else the Python oracle);
  - no dropped carry, lost carry or stale read outside the sites declared in EXEMPT;
  - every call site of a carry primitive in fourq_b200/csrc (a text scan, comments excluded) was executed;
  - every start and middle site produced carry-out 0 and 1, every middle and end site read carry-in 0 and 1, except the
    (site, value) pairs of EXEMPT, whose value must then really never occur;
  - forcing the carry-in of any site that read a 1 to 0 changes at least one corpus row."""
import ctypes
import os
import re
import subprocess
import time

import numpy as np
import pytest

import carry_corpus

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "fourq_b200", "csrc")
START = ("add_cc", "sub_cc", "mad_lo_cc")
MIDDLE = ("addc_cc", "subc_cc", "madc_lo_cc", "madc_hi_cc")
END = ("addc", "subc", "madc_hi")
PRIMS = START + MIDDLE + END
KIND = {name: i for i, name in enumerate(PRIMS)}             # arith.cuh fqsim::CarryKind order

# (file, function, call text) -> {what cannot happen there: reason}.  "cout1" = the site never carries out, "cin1" = it never
# reads a carry of 1, "dropped" = an end op whose wrap is the intent (a borrow turned into a mask).
EXEMPT = {
    ("fp.cuh", "fp_sqr", "addc_cc(O5, 0)"): {
        "cout1": "O5 = lo(a2 e3) is even (e3 = 2 a3), so O5 + 1 < 2^32"},
    ("fp.cuh", "fp_sqr", "addc(O6, 0)"): {
        "cin1": "reads the carry of addc_cc(O5, 0), which cannot carry (O5 is even)"},
    ("x25519.cuh", "f25_sqr", "add_cc(E[1], O[0])"): {
        "cout1": "E[1] is never written: no product a_i a_j with i < j sits at limb position 0 or 1 of the even lattice"},
    ("x25519.cuh", "f25_sqr", "addc(E[15], O[14])"): {
        "cin1": "the cross sum c = sum a_i a_j W^(i+j) (i < j, W = 2^32) is < W^13 (W^2 - 3 + 2/W) < W^15: nothing reaches limb 15"},
    ("x25519.cuh", "f25_sqr", "add_cc(m[0], s[0])"): {
        "cout1": "m[0] = 2 c[0] = 0: the cross sum has no limb 0"},
    ("x25519.cuh", "f25_sub", "subc(0, 0)"): {
        "dropped": "carry extraction: 0 - 0 - borrow is the all-ones mask of a borrow"},
    ("scalar.cuh", "scal_reduce_odd", "subc(0, 0)"): {
        "dropped": "carry extraction: 0 - 0 - borrow is the all-ones mask of a borrow"},
}


# ---------------------------------------------------------------- the call sites in the sources

_CALL = re.compile(r"\b(" + "|".join(PRIMS) + r")\(")
_FUNC = re.compile(r"^(?:template\s*<[^>]*>\s*)?[A-Za-z_][\w\s\*&:<>,]*?\b(\w+)\s*\(")


def _strip_comments(text):
    """The text with comments blanked out (same line and column numbers)."""
    out = re.sub(r"/\*.*?\*/", lambda m: re.sub(r"[^\n]", " ", m.group(0)), text, flags=re.S)
    return "\n".join(re.sub(r"//.*", "", line) for line in out.split("\n"))


def _call_text(line, start):
    depth = 0
    for i in range(start, len(line)):
        depth += line[i] == "("
        depth -= line[i] == ")"
        if line[i] == ")" and depth == 0:
            return line[start:i + 1]
    raise AssertionError("call spans lines: " + line)


def source_sites():
    """{(file, line, column of the '('): (function, call text, primitive)} for every call of a carry primitive in csrc."""
    sites = {}
    for f in sorted(os.listdir(CSRC)):
        if not f.endswith((".cuh", ".cu", ".h")):
            continue
        lines = _strip_comments(open(os.path.join(CSRC, f)).read()).split("\n")
        func = None
        for no, line in enumerate(lines, 1):
            if line[:1].isalpha() and not line.startswith(("struct", "typedef", "enum", "namespace")):
                m = _FUNC.match(line)
                if m:
                    func = m.group(1)
            for m in _CALL.finditer(line):
                if func == m.group(1) and f == "arith.cuh":
                    continue                                            # the definition itself
                sites[(f, no, m.end())] = (func, _call_text(line, m.start()), m.group(1))
    return sites


# ---------------------------------------------------------------- the sanitizer build

@pytest.fixture(scope="module")
def tracer():
    so = os.path.join(HERE, "hostsim", "libfq_hostsim_carry.so")
    srcs = [os.path.join(HERE, "hostsim", f) for f in ("hostsim.cpp", "carry_trace.cpp", "build_carry.sh")] + [
        os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call([os.path.join(HERE, "hostsim", "build_carry.sh")])
    lib = ctypes.CDLL(so)
    lib.carry_dump.restype = ctypes.c_size_t
    lib.carry_dump.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
    lib.carry_force_site.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    return lib


def dump(lib):
    n = lib.carry_dump(None, 0)
    buf = ctypes.create_string_buffer(n)
    lib.carry_dump(buf, n)
    out = {}
    for row in buf.value.decode().splitlines():
        f, line, col, kind, *c = row.split("\t")
        out[(f, int(line), int(col))] = [int(kind)] + [int(x) for x in c]
    return out          # site -> [kind, calls, cin0, cin1, cout0, cout1, dropped, lost, stale]


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


FP2 = {"mul": 0, "sqr": 1, "inv": 2, "add": 3, "sub": 4, "neg": 5, "conj": 6}
FP = {"mul": 0, "sqr": 1, "inv": 2, "add": 3, "sub": 4, "neg": 5, "invsqrt": 6}
F25 = {"mul": 0, "sqr": 1, "inv": 2, "add": 3, "sub": 4}
ROWS = 16                                                       # batchinv.cuh FQ_BATCHINV_ROWS, as the GPU kernels run


def simulate(lib, rs):
    """The rows of rs through the simulation function that models its GPU entry point: (out, status or None)."""
    op, ins, n = rs.op, rs.ins, ctypes.c_size_t(rs.n)
    a = ins[0]; b = ins[1] if len(ins) > 1 else None
    kind, _, name = op.partition("_")
    st = None
    if op in ("fp2_select",):
        out = np.zeros_like(a)
        assert lib.sim_select(2, _p(ins[2]), _p(a), _p(b), _p(out), n) == 0
    elif op == "fp2_inv":
        out = np.zeros_like(a)
        assert lib.sim_fp2_inv_batched(_p(a), _p(out), n, ROWS) == 0
    elif op == "fp2_invsqrt":
        out = np.zeros_like(a)
        assert lib.sim_fp2_invsqrt(_p(a), _p(out), n) == 0
    elif kind == "fp2":
        out = np.zeros_like(a)
        assert lib.sim_fp2_op(FP2[name], _p(a), _p(b), _p(out), n) == 0
    elif kind == "fp":
        out = np.zeros_like(a)
        assert lib.sim_fp_row_op(FP[name], _p(a), _p(b), _p(out), n) == 0
    elif op == "f25519_inv":
        out = np.zeros_like(a)
        assert lib.sim_f25_inv_batched(_p(a), _p(out), n, ROWS) == 0
    elif kind == "f25519":
        out = np.zeros_like(a)
        assert lib.sim_f25_op(F25[name], _p(a), _p(b), _p(out), n) == 0
    elif op == "x25519":
        out = np.zeros_like(a)
        assert lib.sim_x25519_batched(_p(a), _p(b), _p(out), n, ROWS) == 0
    elif op == "decode":
        out = np.zeros((rs.n, 64), np.uint8); st = np.zeros(rs.n, np.uint8)
        assert lib.sim_decode(_p(a), _p(out), _p(st), n) == 0
    elif op in ("mul_base", "mul_endo_base"):
        out = np.zeros((rs.n, 32), np.uint8)
        assert lib.sim_fixed_base(2 if op == "mul_endo_base" else 0, _p(a), _p(out), None, n) == 0
    elif op == "dh_endo":
        out = np.zeros((rs.n, 32), np.uint8); st = np.zeros(rs.n, np.uint8)
        assert lib.sim_dh_endo(_p(a), _p(b), _p(out), _p(st), n) == 0
    else:
        raise AssertionError(op)
    return out, st


def _agree(got, want):
    return (got[0] == want[0]).all(axis=1) & (True if want[1] is None else got[1] == want[1])


# ---------------------------------------------------------------- the checks

@pytest.fixture(scope="module")
def run(tracer):
    """Every row set once through the sanitizer: per row set its site counters and whether each row equals its reference."""
    sets = carry_corpus.build()
    per_set, mism = {}, {}
    tracer.carry_force_site(None, 0, 0, -1)
    for rs in sets:
        tracer.carry_reset()
        got = simulate(tracer, rs)
        per_set[rs.name] = dump(tracer)
        rs.want = carry_corpus.reference(rs)
        ok = _agree(got, rs.want)
        if not ok.all():
            mism[rs.name] = [bytes(x).hex() for x in rs.ins[0][~ok][:3]]
    total = {}
    for counts in per_set.values():
        for site, c in counts.items():
            t = total.setdefault(site, [c[0]] + [0] * (len(c) - 1))
            for i in range(1, len(c)):
                t[i] += c[i]
    return sets, per_set, total, mism


def _exempt(sites):
    """{site: {what: reason}} of EXEMPT: each key stands for every call with that text in that function (at least one)"""
    out = {}
    for (f, func, text), what in EXEMPT.items():
        hits = [s for s, (fn, t, _) in sites.items() if s[0] == f and fn == func and t == text]
        assert hits, ("EXEMPT entry matches no call site", f, func, text)
        for h in hits:
            out[h] = what
    return out


def test_corpus_rows_equal_reference(run):
    assert not run[3], run[3]


def test_no_carry_rule_fires(run):
    sites = source_sites()
    ex = _exempt(sites)
    bad = []
    for site, c in run[2].items():
        for rule, v in (("dropped", c[6]), ("lost", c[7]), ("stale", c[8])):
            if v and rule not in ex.get(site, {}):
                bad.append((rule, site, sites.get(site), v))
    assert not bad, bad


def test_every_site_executed_and_covered_both_ways(run):
    sites = source_sites()
    ex = _exempt(sites)
    total = run[2]
    assert set(total) <= set(sites), sorted(set(total) - set(sites))          # the scan sees every site the simulation runs
    missing = sorted(set(sites) - set(total))
    assert not missing, [(s, sites[s]) for s in missing]
    gaps, stale_ex = [], []
    covered = 0
    for site, (func, text, prim) in sorted(sites.items()):
        c = total[site]
        assert c[0] == KIND[prim], (site, c[0], prim)
        need = []
        if prim in START + MIDDLE:
            need += [("cout0", c[4]), ("cout1", c[5])]
        if prim in MIDDLE + END:
            need += [("cin0", c[2]), ("cin1", c[3])]
        e = ex.get(site, {})
        for what, v in need:
            if what in e:
                if v:
                    stale_ex.append((site, func, text, what, v))            # an exemption whose value does occur: the table is wrong
            elif not v:
                gaps.append((site, func, text, what))
        covered += all(v or what in e for what, v in need)
    print("\ncarry sites: %d in the sources, %d executed, %d covered both ways (exemptions included)" % (len(sites), len(total), covered))
    for site, what in sorted(ex.items()):
        for k, reason in what.items():
            print("  exempt %s:%d %s %s: %s" % (site[0], site[1], sites[site][1], k, reason))
    assert not stale_ex, stale_ex
    assert not gaps, gaps


def test_forcing_any_carry_in_of_one_to_zero_changes_a_row(run, tracer):
    """Mutation check: each site that read a carry of 1 is forced to read 0; the row set that exercised it the least expensively
    must then give at least one row different from its reference."""
    sets, per_set, total, _ = run
    by_name = {rs.name: rs for rs in sets}
    cost = {rs.name: rs.n * (1000 if rs.op in ("x25519", "mul_base", "mul_endo_base", "dh_endo", "decode") or rs.op.endswith("inv")
                             or rs.op.endswith("invsqrt") else 1) for rs in sets}
    survivors = []
    t0 = time.time()
    try:
        for site in sorted(s for s, c in total.items() if c[3]):
            names = sorted((n for n, c in per_set.items() if site in c and c[site][3]), key=cost.get)
            tracer.carry_force_site(site[0].encode(), site[1], site[2], 0)
            for name in names:
                rs = by_name[name]
                if not _agree(simulate(tracer, rs), rs.want).all():
                    break
            else:
                survivors.append(site)
    finally:
        tracer.carry_force_site(None, 0, 0, -1)
    print("\nmutation check: %d sites forced, %.1f s" % (sum(1 for c in total.values() if c[3]), time.time() - t0))
    assert not survivors, [(s, source_sites().get(s)) for s in survivors]
