"""Pin the C restatement (oracle/scan_oracle.c) on the golden vectors generated
from the unmodified reference (tests/golden/make_golden.py).  CPU only."""
import json
import os

import numpy as np
import pytest

from oracles import WINDOWS, fnv1a_int64
from scan_cases import expected, make_reads

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def gold():
    vec = np.load(os.path.join(GOLD, "ref_vectors.npz"))
    with open(os.path.join(GOLD, "ref_vectors.json")) as f:
        meta = json.load(f)
    return vec, meta


def test_sine_tables(port_oracle, gold):
    vec, _ = gold
    for m in (1, 2, 3, 4, 5, 6, 8, 10, 12):
        assert np.array_equal(port_oracle.sine_table(m), vec[f"sine_{m}"])


def test_window_tables(port_oracle, gold):
    vec, _ = gold
    for w in WINDOWS:
        for n in (32, 1024):
            assert np.array_equal(port_oracle.window_coefs(w, n), vec[f"win_{w}_{n}"]), (w, n)


def test_fix_fft(port_oracle, gold):
    vec, meta = gold
    for c in meta["fix_fft"]:
        got = port_oracle.fix_fft(vec[c["key"] + "_in"], c["m"])
        assert np.array_equal(got, vec[c["key"] + "_out"]), c


def test_fix_mpy_closed_form(port_oracle):
    """(a*b + 2^14) >> 15 equals the reference's two-step FIX_MPY (rtl_power.c:263-269)."""
    rng = np.random.default_rng(0)
    a = rng.integers(-32768, 32768, 200000).astype(np.int64)
    b = rng.integers(-32768, 32768, 200000).astype(np.int64)
    c = (a * b) >> 14
    two_step = ((c >> 1) + (c & 1)).astype(np.int16)
    closed = ((a * b + 16384) >> 15).astype(np.int16)
    assert np.array_equal(two_step, closed)
    for x, y in [(-32768, -32768), (32767, 32767), (-16384, 1), (16383, -32768), (0, 5)]:
        assert port_oracle.lib.oracle_fix_mpy(x, y) == int(np.array((x * y + 16384) >> 15).astype(np.int16))


def test_decimators_and_dc(port_oracle, gold):
    vec, meta = gold
    for c in meta["fifth_order"]:
        assert np.array_equal(port_oracle.fifth_order(vec[c["key"] + "_in"], c["length"]), vec[c["key"] + "_out"]), c
    for c in meta["generic_fir"]:
        assert np.array_equal(port_oracle.generic_fir(vec[c["key"] + "_in"], c["length"], c["table"]),
                              vec[c["key"] + "_out"]), c
    for c in meta["remove_dc"]:
        assert np.array_equal(port_oracle.remove_dc(vec[c["key"] + "_in"], c["length"]), vec[c["key"] + "_out"]), c


def test_rms(port_oracle, gold):
    from oracles import synth_bytes
    _, meta = gold
    for c in meta["rms"]:
        b = synth_bytes(port_oracle.lib, c["mode"], c["seed"], c["param"], 1, 0, 0, 16384)
        assert port_oracle.rms_power(b, 1234, 0) == c["sum"]
        assert port_oracle.rms_power(b, 10**9, 1) == c["peak"]


def test_scans_and_csv_rows(port_oracle, gold):
    """whole hop visits + the text rows csv_dbm printed for them; the host planner's whole plan == the reference's"""
    from rtlsdr_b200.planner import plan_scan
    vec, meta = gold
    for c in meta["scan"]:
        plan = dict(c["plan"])
        plan["peak_hold"] = c["peak"]
        w = port_oracle.window_coefs(c["window"], 1 << plan["bin_e"])
        reads, hops = make_reads(port_oracle.lib, plan, c["passes"], c["mode"], c["seed"], c["param"])
        avg, smp, db = expected(port_oracle, plan, w, reads, hops)
        assert np.array_equal(avg, vec[c["key"] + "_avg"]), c["freq"]
        assert np.array_equal(smp, vec[c["key"] + "_samples"])
        p = plan_scan(c["freq"], c["crop"], None if c["fir"] < 0 else c["fir"])
        mine = p.as_dict()
        for k, v in c["plan"].items():
            assert mine[k] == v, (c["freq"], k, mine[k], v)
        for h in range(plan["tune_count"]):
            assert p.csv_row(h, int(smp[h]), db[h]) == c["csv"][h], (c["freq"], h)


def test_known_answer_hashes(port_oracle):
    """SURVEY.md 8(c) rows, all of them (about a second of CPU): the 2^17-bin row checks the restatement's large
    fix_fft, the 512 / 623-hop rows the wideband plans, against the reference's own bins."""
    from rtlsdr_b200.planner import plan_scan
    with open(os.path.join(GOLD, "kat.json")) as f:
        kat = json.load(f)
    assert len(kat) == 11
    for c in kat:
        plan = plan_scan(c["freq"], c["crop"], None if c["fir"] < 0 else c["fir"]).as_dict()
        plan["peak_hold"] = c["peak"]
        w = port_oracle.window_coefs(c["window"], 1 << plan["bin_e"])
        reads, hops = make_reads(port_oracle.lib, plan, c["passes"], c["mode"], 0, 0)
        avg, smp, _ = expected(port_oracle, plan, w, reads, hops)
        assert f"{fnv1a_int64(avg):016x}" == c["fnv"], c
        assert int(smp[0]) == c["samples0"]
        assert [int(v) for v in avg[0][:3]] == c["avg0_head"]
