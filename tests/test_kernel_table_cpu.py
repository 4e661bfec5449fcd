"""The kernel table of csrc/wshmpc.cu (one row per large kernel and translation unit), read as text: no GPU and no nvcc."""
import os
import re

import __graft_entry__ as g

SRC = os.path.join(g.CSRC, 'wshmpc.cu')
ROW = re.compile(r'^#define WS_ROW_(\d+)\(X\)\s+X\(([^)]*)\)\s*$', re.M)


def rows():
    """[(unit, name, family, lanes, rule, plant, fb)] of the table, as written"""
    with open(SRC) as f:
        text = f.read()
    out = []
    for u, body in ROW.findall(text):
        cols = [c.strip() for c in body.split(',')]
        assert len(cols) == 7 and cols[0] == u, (u, cols)
        out.append((int(u),) + tuple(cols[1:]))
    assert out, 'no kernel table in ' + SRC
    return out, text


def test_units_are_one_to_n():
    table, _ = rows()
    assert [r[0] for r in table] == list(range(1, len(table) + 1))


def test_every_row_is_listed_once():
    table, text = rows()
    listing = re.search(r'^#define WS_KERNELS\(X\)((?:.*\\\n)*.*)$', text, re.M).group(1)
    assert re.findall(r'WS_ROW_(\d+)\(X\)', listing) == [str(r[0]) for r in table]


def test_names_and_variants_are_unique():
    table, _ = rows()
    assert len({r[1] for r in table}) == len(table)
    assert len({(fam, lanes, rule != '0', plant, fb) for _, _, fam, lanes, rule, plant, fb in table}) == len(table)
    assert {r[2] for r in table} == {'K1', 'BNB', 'LOOP'}
    assert {r[3] for r in table} == {'1', 'WS_MAXL'}


def test_one_lane_kernels_take_the_odd_units():
    """WS_WIDE_REGS (csrc/qp_device.cuh) gives the odd units 255 registers per thread"""
    table, _ = rows()
    for u, name, _, lanes, *_ in table:
        assert (lanes == '1') == (u % 2 == 1), (u, name, lanes)
        assert name.endswith('_1' if lanes == '1' else '_m'), (u, name)


def test_build_compiles_one_unit_per_row(tmp_path, monkeypatch):
    table, _ = rows()
    calls = []
    monkeypatch.setattr(g.subprocess, 'check_call', lambda cmd: calls.append(cmd))
    g.compile_library(str(tmp_path / 'lib.so'), objdir=str(tmp_path))
    units = sorted(int(a[len('-DWS_TU='):]) for cmd in calls for a in cmd if a.startswith('-DWS_TU='))
    assert units == list(range(len(table) + 1))
    assert sum(a.endswith('.o') for a in calls[-1]) == len(table) + 1      # the link takes every unit
