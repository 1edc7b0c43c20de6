"""The repair rounds of the entropy stage on scans that never self-synchronise (sync_adversary.py), on the CPU: the
oracle decodes every generated file to the generator's coefficients, and the simulation of the kernels decodes it
exactly under the planner settings of the GPU tests, with diagnostics that prove the input adversarial."""
import functools
import itertools

import numpy as np
import pytest

import oracle_ffi as O
import sim_ffi as S
import sync_adversary as A


@functools.lru_cache(maxsize=None)
def _corpus(small):
    return A.corpus(small)


def _ext(case):
    return O.EXT_DRI if case.ri else O.EXT_NONE


def _same(got, want):
    return len(got) == len(want) and all(np.array_equal(a, w) for a, w in zip(got, want))


@functools.lru_cache(maxsize=None)
def _oracle(small, i):
    c = _corpus(small)[i]
    o = O.decode(c.file, layout=O.LAYOUT_SPEC, ext=_ext(c))
    return o.status, o.bytes_read, o.coefs, o.scan_len


@pytest.mark.parametrize("small", [True, False])
def test_oracle_decodes_the_generated_coefficients(small):
    """The oracle's coefficients are the generator's; without DRI it reads every byte of the entropy-coded data
    (counted after unstuffing) and stops at the EOI, as on the encoder's files (the reference that the simulation's and the device's bytes_read are
    held to)."""
    for i, c in enumerate(_corpus(small)):
        status, bytes_read, coefs, scan_len = _oracle(small, i)
        assert status == 0, c.name
        assert _same(coefs, c.want), c.name
        if not c.ri:
            assert bytes_read == A.scan_bits(c.file) // 8, (c.name, bytes_read)   # bytes after unstuffing
            assert scan_len - bytes_read == 2, (c.name, scan_len, bytes_read)


def _sim(case, sub_bits):
    (r,), d = S.decode_batch([case.file], ext=_ext(case), sub_bits=sub_bits)
    return r, d


def _check_sim(small, i, r):
    c = _corpus(small)[i]
    status, bytes_read, _, _ = _oracle(small, i)
    assert r.status == 0, (c.name, r.status)
    assert _same(r.coefs, c.want), f"{c.name}: coefficients differ"
    if not c.ri:
        assert r.bytes_read == bytes_read, (c.name, r.bytes_read, bytes_read)


def test_the_corpus_drives_the_repair_rounds(capsys):
    """Full size, 1024-bit subsequences, the planner's look-back: the zigzag chain needs nsub - 2 rounds or more (one
    link per round), the crowds and the chain-then-crowd files find more than 256 broken links in each of at least 200
    rounds, and no file needs more than nsub - 1 rounds: the bound verify_scan_kernel's loop relies on."""
    lines = []
    for i, c in enumerate(_corpus(False)):
        r, d = _sim(c, 1024)
        _check_sim(False, i, r)
        n = A.nsub(c.file, 1024)
        lines.append(f"{c.name:24s} nsub {n:5d}  repair rounds {d['repair_iters']:5d}  most broken links in a round "
                     f"{d['max_broken']:5d}  rounds with more than 256 {d['crowded_rounds']:5d}  repairs {d['repairs']}")
        assert d["repair_iters"] <= n - 1, c.name
        if c.kind == "chain":
            assert d["repair_iters"] >= n - 2 and d["max_broken"] == 1, c.name
        if c.kind in ("crowd", "chain_crowd"):
            assert n >= 1024 and d["max_broken"] > 256 and d["crowded_rounds"] >= 200, c.name
        if c.kind == "chain_crowd":
            assert d["repair_iters"] >= n - 2, c.name
    with capsys.disabled():
        print("\n" + "\n".join(lines))


def test_restart_interval_files_drive_repairs(monkeypatch):
    """With the synchronisation pass forced (JPGPU_INTERVAL_MODE=0) and no look-back, the DRI files need repair
    rounds too: every marker restores the phase, but the cold starts between markers still land on wrong phases.
    (With the planner's look-back of 8192 bits, longer than their intervals, every cold start crosses a marker.)"""
    monkeypatch.setenv("JPGPU_INTERVAL_MODE", "0")
    monkeypatch.setenv("JPGPU_LOOKBACK_BITS", "0")
    for i, c in enumerate(_corpus(False)):
        if not c.ri:
            continue
        r, d = _sim(c, 1024)
        _check_sim(False, i, r)
        assert d["repair_iters"] > 0 and d["max_broken"] > 0, (c.name, d)


def test_settings_cover_every_pair():
    rows = A.settings()
    assert len(rows) == 16
    for a, b in itertools.combinations(rows[0], 2):
        want = {(x, y) for x in {r[a] for r in rows} for y in {r[b] for r in rows}}
        assert {(r[a], r[b]) for r in rows} == want, (a, b)


@pytest.mark.parametrize("row", A.settings(), ids=A.settings_id)
def test_simulation_decodes_the_corpus_exactly(row, monkeypatch):
    """The small corpus under every row of the settings array (the simulation has one multi-symbol switch for the
    synchronisation pass and the repair walks: JPGPU_SYNC_MULTI)."""
    A.apply(monkeypatch, row)
    S.set_sync_multi(row["JPGPU_SYNC_MULTI"] == "1")
    try:
        sub_bits = int(row["JPGPU_SUBSEQ_BITS"])
        for i, c in enumerate(_corpus(True)):
            r, d = _sim(c, sub_bits)
            _check_sim(True, i, r)
            assert d["repair_iters"] <= max(1, A.nsub(c.file, sub_bits) - 1), c.name
    finally:
        S.set_sync_multi(True)


@pytest.mark.parametrize("sub_bits", [1024, 2048])
def test_multi_symbol_sync_records_equal_the_single_symbol_ones(sub_bits):
    """The synchronisation records (digest over every SubInfo / SegRec before the repairs) of the multi-symbol pass
    equal the symbol-by-symbol ones on the adversarial corpus, as on natural files."""
    cases = [c for c in _corpus(True) if not c.ri]
    try:
        S.set_sync_multi(True)
        a, da = S.decode_batch([c.file for c in cases], sub_bits=sub_bits)
        S.set_sync_multi(False)
        b, db = S.decode_batch([c.file for c in cases], sub_bits=sub_bits)
    finally:
        S.set_sync_multi(True)
    assert da["sync_digest"] == db["sync_digest"]
    assert da["repairs"] == db["repairs"] and da["repair_iters"] == db["repair_iters"]
    for c, x, y in zip(cases, a, b):
        assert x.status == y.status == 0 and _same(x.coefs, c.want) and _same(y.coefs, c.want), c.name

