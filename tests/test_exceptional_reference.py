"""The fixtures of tests/test_gpu_exceptional.py, checked on the CPU.

The structured oracle (bitwise the reference's arithmetic) is driven line by line with the policy of include/ekf.h: a
pair whose S is singular is no match.  Its own LU (ekfo_gate_pair: S^-1 = 0 exactly when a diagonal entry of U is zero)
must find exactly the pairs the fixture meant to be singular singular -- in every line of every scan, also after
earlier matches in the same scan -- and every other pair regular.  The extended-precision reference must then give the
same associations, line counts and statuses, with no gate decision near the threshold.
"""
import ctypes

import numpy as np
import pytest

import hp_reference as hp
import test_gpu_exceptional as t

SMALL = ["sing_small", "sing_past", "rank1", "all_sing", "cap_small", "cap_reset", "both_small"]
BIG = ["sing_big", "past_big", "cap_big", "cap_big_reset", "chunk_cap2", "chunk_cap3"]


def _oracle_from(y, P, L, cap, headroom):
    from oracle.oracle import StructuredOracle
    so = StructuredOracle(cap, reset_headroom=headroom)
    np.ctypeslib.as_array(so._lib.ekfo_y_ptr(so._h), shape=(so.n,))[:] = y
    so.P_view()[:] = P
    so._lib.ekfo_set_lines(so._h, ctypes.c_int(L))
    so.set_pose(y[:3])
    return so


def drive_oracle(so, scans, sing):
    """Runs `scans` on the oracle with singular pairs skipped.  `sing`: the landmarks meant to be singular (angle of zero
    variance); lines with R_SING make them singular.  Returns [(status, j, L)] and the number of singular pairs seen."""
    sing = set(sing)
    out, n_sing = [], 0
    for s, (u, z, R) in enumerate(scans):
        so.predict(u)
        m = z.shape[0]
        j = np.full(m, -1, np.int32)
        met, L0 = False, so.lines
        matched = set()
        for i in range(m):
            if so.lines == 0:
                so.queue(i)
                continue
            for k in range(so.lines):
                if k in matched:
                    continue
                S, Si, v, d2 = so.gate_pair(k, z[i], R[i])
                singular = not Si.any()
                meant = k in sing and tuple(R[i]) in (t.R_SING, t.R_RANK1)
                assert singular == meant, "scan %d line %d landmark %d: singular %s, meant %s (S = %s)" % (
                    s, i, k, singular, meant, S.tolist())
                if singular:
                    assert S[0, 0] * S[1, 1] - S[0, 1] * S[1, 0] == 0.0
                    met = True; n_sing += 1
                    continue
                if not (np.sqrt(abs(d2)) > 0.4):
                    j[i] = k
                    break
            if j[i] >= 0:
                matched.add(int(j[i]))
                so.update(int(j[i]), z[i], R[i])
            else:
                so.queue(i)
        st = so.end(z, R)
        added = [i for i in range(m) if j[i] < 0][:max(0, so.lines - L0)] if so.lines >= L0 else []
        if so.lines < L0 or (so.lines == 0 and m):       # a map reset
            sing = set()
        else:
            for q, i in enumerate(added):
                if tuple(R[i]) == t.R_SING:
                    sing.add(L0 + q)
        out.append((st if st or not met else 3, j, so.lines))
    return out, n_sing


def _check_case(name):
    c = t.case_inputs(name)
    so = _oracle_from(c["y"], c["P"], c["L"], c["cap"], c["headroom"])
    got, n_sing = drive_oracle(so, c["inputs"], c["sing"])
    so.close()
    ref = t.reference(name)
    for s, ((st, j, L), r) in enumerate(zip(got, ref)):
        assert np.array_equal(j, r["j"]), "%s scan %d: oracle %s, reference %s" % (name, s, j, r["j"])
        assert st == r["st"] and L == r["L"], "%s scan %d: oracle (%d, %d), reference (%d, %d)" % (
            name, s, st, L, r["st"], r["L"])
    return got, n_sing


@pytest.mark.parametrize("name", SMALL)
def test_fixture_pairs_are_exactly_singular(name):
    got, n_sing = _check_case(name)
    st = [g[0] for g in got]
    c = t.CASES[name]
    specs = c["scans"]
    # every case exercises what it is named for, and the scan after the branch is clean
    if name in ("sing_small", "all_sing"):
        assert 3 in st and st[-1] == 0 and n_sing >= 4
    if name == "sing_past":
        assert st == [0, 3, 3] and got[0][1].tolist() == [0] and got[2][1].tolist() == [0, 2]   # 1, 4 past the winner
    if name == "rank1":
        assert st == [3, 0, 3] and got[0][1].tolist() == [2, 0] and got[2][1].tolist() == [5, -1] and n_sing >= 3
    if name == "cap_small":
        assert st == [2, 2, 0] and [g[2] for g in got] == [13, 13, 13]
    if name == "both_small":
        assert st == [2, 3, 0] and n_sing >= 2
    if name == "sing_small":
        j0 = got[0][1]
        assert j0[0] == 2 and j0[1] == -1 and j0[2] == 4 and j0[3] == 6       # first fit skips 1, then matches 2
        assert got[2][1][1] == 8 and got[2][1][0] == 1
    if name == "all_sing":
        assert all((g[1] == -1).all() for g in got[:2]) and got[1][2] == 6 + 4 + 3
    if name == "cap_reset":
        assert st[0] == 2 and got[0][2] == 0                                   # the reset follows the drop
    assert len(specs) == len(got)


@pytest.mark.parametrize("name", BIG)
def test_big_fixtures(name):
    got, n_sing = _check_case(name)
    st = [g[0] for g in got]
    c = t.CASES[name]
    if name.startswith("chunk"):
        assert st[0] == 2 and got[0][2] == c["cap"] and st[1] == 0 and n_sing > 0
        first_drop = [i for i in range(40) if got[0][1][i] < 0][c["cap"] - c["L"]]
        assert first_drop // 16 == (1 if name == "chunk_cap2" else 2), first_drop
        assert (got[0][1][:len([s for s in c["scans"][0] if s[0] == "m"])] >= 0).all()
    elif name == "sing_big":
        assert st == [3, 0, 3, 0] and got[0][1].tolist() == [2, -1, 4, 6]
    elif name == "past_big":
        assert st == [0, 3, 3] and got[0][1].tolist() == [0]
    elif name == "cap_big":
        assert st == [2, 2, 0] and got[-1][2] == c["cap"]
    else:
        assert st[0] == 2 and got[0][2] == 0


def test_batch_fixtures():
    """Every batch filter, seeded from the empty map, against the oracle: the landmarks appended with R00 = R01 = 0 are
    exactly singular with the R_SING lines, and the steps' statuses aggregate as ekf_batch_collect does."""
    from oracle.oracle import StructuredOracle
    for kind, headroom in (("small", 0), ("small", 1), ("rounds", 0)):
        c = t.BATCHES[kind]
        scans = t.batch_inputs(kind)
        ref, states = t.batch_reference(kind, headroom)
        per = []
        for f in range(len(c["sing"])):
            so = StructuredOracle(c["cap"], reset_headroom=headroom)
            got, _ = drive_oracle(so, [(u[f], z[f], R[f]) for (u, z, R) in scans], ())
            so.close()
            per.append(got)
        for s, r in enumerate(ref):
            assert [p[s][0] for p in per] == r["fst"], (headroom, s)
            assert np.array_equal(np.stack([p[s][1] for p in per]), r["j"]), (headroom, s)
        if kind == "small" and headroom == 0:
            assert [r["st"] for r in ref] == [0, 2, 3, 0, 2]
            assert ref[1]["fst"] == [3, 0, 2, 2] and ref[3]["j"][0].tolist() == [0, 8]   # singular pairs past 0: clean
        if kind == "rounds":
            # f0 gates 40 singular pairs (two rounds of full gates) before its winner; f1's singular pairs lie past it
            assert [r["fst"] for r in ref[1:]] == [[3, 0], [0, 0], [3, 0]]
            assert ref[1]["j"].tolist() == [[50, 60], [5, 6]] and ref[3]["j"].tolist() == [[45], [45]]

