"""The best-matches searches (cds_search_best_matches and the streamed variants): exported symbols, the ctypes layout of
cds_target_groups, the TargetGroups helper and the argument checks that run before any device is touched."""
import ctypes as C
import os
import re

import numpy as np

from colormipsearch_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("cds_search_best_matches", "cds_search_stream_best_matches_tiff", "cds_search_stream_best_matches_rgb",
       "cds_debug_select_best_matches_device")


def test_new_symbols_are_exported():
    L = capi.lib()
    for name in NEW:
        assert hasattr(L, name), name


def test_target_groups_struct_follows_the_header():
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "cdsgpu.h")).read(), flags=re.S)
    body = re.search(r"typedef struct cds_target_groups \{(.*?)\} cds_target_groups;", header, flags=re.S).group(1)
    want = []
    for decl in filter(None, (d.strip() for d in body.split(";"))):
        name = decl.split()[-1].lstrip("*")
        want.append((name, C.sizeof(C.c_void_p) if "*" in decl else 4))
    got = [(n, C.sizeof(t)) for n, t in capi.TargetGroupsC._fields_]
    assert got == want
    assert C.sizeof(capi.TargetGroupsC) == 48


def test_target_groups_ids_and_hashes_match_select_best_matches():
    lines = ["R10G01", "", "R10G01", "VT0042", "  ", "UNKNOWN", "R11A02"]
    samples = ["s1", "s2", "s1", "s3", "s2", "s4", "s5"]
    g = capi.TargetGroups(lines, samples)
    assert g.line.tolist() == [0, 1, 0, 2, 1, 1, 3]             # blank -> "UNKNOWN", which is also a key of its own
    assert g.sample.tolist() == [0, 1, 0, 2, 1, 3, 4]
    assert g.line_hash.tolist() == [capi.java_string_hash(s) for s in ("R10G01", "UNKNOWN", "VT0042", "R11A02")]
    assert g.sample_hash.tolist() == [capi.java_string_hash(s) for s in ("s1", "s2", "s3", "s4", "s5")]
    lid, lhash = capi._group_ids(lines)
    assert np.array_equal(lid, g.line) and np.array_equal(lhash, g.line_hash)
    s = g.struct()
    assert s.n_lines == 4 and s.n_samples == 5 and s.line[3] == 2 and s.sample_hash[4] == capi.java_string_hash("s5")


def _bad_arg(status):
    assert status == capi.CDS_ERR_BAD_ARG
    return capi.lib().cds_last_error(None).decode()


def _groups(line, sample, n_lines, n_samples):
    line = np.asarray(line, np.int32); sample = np.asarray(sample, np.int32)
    lh = np.arange(max(n_lines, 1), dtype=np.int32); sh = np.arange(max(n_samples, 1), dtype=np.int32)
    keep = (line, sample, lh, sh)
    return capi.TargetGroupsC(line.ctypes.data_as(capi._i32p), sample.ctypes.data_as(capi._i32p), lh.ctypes.data_as(capi._i32p), n_lines,
                              sh.ctypes.data_as(capi._i32p), n_samples), keep


def test_bad_arguments_without_a_device():
    L = capi.lib()
    out32 = np.zeros(4, np.int32); out64 = np.zeros(4, np.int64); out8 = np.zeros(4, np.uint8); cnt = C.c_int64(0)
    tail = (0.0, 300, 1, 1, 4, out32.ctypes.data_as(capi._i32p), out64.ctypes.data_as(capi._i64p), out32.ctypes.data_as(capi._i32p),
            out8.ctypes.data_as(capi._u8p), C.byref(cnt))
    rgb = np.zeros((2, 4, 4, 3), np.uint8)
    blob = np.zeros(8, np.uint8); offs = np.array([0, 4, 8], np.int64)
    # NULL groups
    assert "groups is NULL" in _bad_arg(L.cds_search_stream_best_matches_rgb(None, None, capi._ptr(rgb), 2, None, *tail))
    assert "groups is NULL" in _bad_arg(L.cds_search_stream_best_matches_tiff(None, None, capi._ptr(blob), offs.ctypes.data_as(capi._i64p), 2, None, *tail))
    assert "NULL" in _bad_arg(L.cds_search_best_matches(None, None, None, None, *tail))
    # ids outside their ranges
    for line, sample, nl, ns, what in (([0, 2], [0, 0], 2, 1, "line id 2 of target 1"), ([0, -1], [0, 0], 1, 1, "line id -1"),
                                       ([0, 0], [0, 1], 1, 1, "sample id 1 of target 1"), ([0, 0], [-3, 0], 1, 1, "sample id -3")):
        g, keep = _groups(line, sample, nl, ns)
        assert what in _bad_arg(L.cds_search_stream_best_matches_rgb(None, None, capi._ptr(rgb), 2, C.byref(g), *tail))
        assert what in _bad_arg(L.cds_search_stream_best_matches_tiff(None, None, capi._ptr(blob), offs.ctypes.data_as(capi._i64p), 2, C.byref(g), *tail))
    # the test hook: groups are checked over the targets the list names, and the list must be in encounter order
    g, keep = _groups([0, 0, 5], [0, 0, 0], 2, 1)
    m = np.array([0, 0], np.int32); t = np.array([0, 2], np.int64); s = np.array([5, 4], np.int32); sel = np.zeros(2, np.int64)
    args = lambda mm, tt, ss, gg: (None, mm.ctypes.data_as(capi._i32p), tt.ctypes.data_as(capi._i64p), ss.ctypes.data_as(capi._i32p), None, len(mm),
                                   gg, 0, 0, 0, sel.ctypes.data_as(capi._i64p), C.byref(cnt))
    assert "line id 5 of target 2" in _bad_arg(L.cds_debug_select_best_matches_device(*args(m, t, s, C.byref(g))))
    assert "groups is NULL" in _bad_arg(L.cds_debug_select_best_matches_device(*args(m, t, s, None)))
    g2, keep2 = _groups([0, 1, 1], [0, 0, 0], 2, 1)
    assert "not sorted" in _bad_arg(L.cds_debug_select_best_matches_device(*args(m, t, s[::-1].copy(), C.byref(g2))))
    assert "not sorted" in _bad_arg(L.cds_debug_select_best_matches_device(*args(m[::-1].copy() + np.array([1, 0], np.int32), t, s, C.byref(g2))))
    # a valid request without a context
    assert "NULL ctx" in _bad_arg(L.cds_debug_select_best_matches_device(*args(m, t, s, C.byref(g2))))


def test_best_list_bytes_is_a_documented_option():
    header = open(os.path.join(ROOT, "include", "cdsgpu.h")).read()
    doc = header[header.index("Tuning / test switches"):header.index("cds_status cds_ctx_set_option")]
    assert '"best_list_bytes"' in doc

