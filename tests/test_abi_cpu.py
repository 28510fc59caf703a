"""CPU checks of the drop-in boundary: the shared library loads and exports every
symbol include/tombo_b200.h declares (no compute calls without a GPU)."""
import ctypes
import os
import re

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    src = open(os.path.join(REPO, 'include', 'tombo_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(tb2_[a-z0-9_]+)\s*\(', src)))


def test_library_loads_and_exports_declared_symbols():
    from tombo_b200 import _lib
    lib = _lib.load()
    assert lib.tb2_abi_version() == 1
    names = declared_functions()
    assert len(names) >= 10
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_status_messages_match_reference_strings():
    from tombo_b200 import _lib
    import oracle
    for st in list(range(0, 22)):
        assert _lib.status_message(st) == oracle.status_message(st)


def test_no_cpu_fallback_without_device():
    from tombo_b200 import _lib
    if _lib.load().tb2_device_count() > 0:
        pytest.skip('a device is present')
    with pytest.raises(_lib.TomboB200Error):
        _lib.Context(0)


def test_python_api_surface_imports_without_gpu():
    from tombo_b200 import tombo_helper as th, tombo_stats as ts, resquiggle as rsq
    for name in ('resquiggle_read', 'segment_signal', 'find_adaptive_base_assignment',
                 'resolve_skipped_bases_with_raw', 'find_seq_start_in_events',
                 'find_static_base_assignment', 'resquiggle_reads'):
        assert callable(getattr(rsq, name))
    for name in ('TomboModel', 'AltModel', 'normalize_raw_signal', 'compute_base_means',
                 'get_read_seg_score', 'calc_kmer_fitted_shift_scale',
                 'load_resquiggle_parameters', 'compute_num_events',
                 'compute_alt_model_read_stats'):
        assert hasattr(ts, name)
    p = ts.load_resquiggle_parameters(th.seqSampleType('DNA', False))
    assert p.bandwidth == 300 and p.start_bw == 750 and p.z_shift > 4.99
    sp = ts.load_resquiggle_parameters(th.seqSampleType('RNA', True), use_save_bandwidth=True)
    assert sp.bandwidth == 1500 and sp.use_t_test_seg
    assert ts.compute_num_events(4300, 444, 5) == 860
    m = th.TomboMotif('CCWGG', 2)
    assert m.motif_pat.pattern == 'CC[AT]GG' and m.mod_base == 'C'


def test_parameters_and_namedtuples_match_reference_when_available():
    """against the reference's values, recorded by tests/golden/make_reference_api_golden.py"""
    import ast
    import json
    from tombo_b200 import tombo_helper as th, tombo_stats as ts, _default_parameters as dp
    g = json.load(open(os.path.join(REPO, 'tests', 'golden', 'reference_api.json')))
    ref = {n: ast.literal_eval(v) for n, v in g['default_parameters'].items()}
    for name in dir(dp):
        if name.isupper():
            assert name in ref and getattr(dp, name) == ref[name], name
    assert len(g['namedtuple_fields']) == 10
    for nt, fields in g['namedtuple_fields'].items():
        assert getattr(th, nt)._fields == tuple(fields), nt
    assert len(g['resquiggle_parameters']) == 4
    for kind, save, b in g['resquiggle_parameters']:
        sst = th.seqSampleType(kind, kind == 'RNA')
        a = ts.load_resquiggle_parameters(sst, use_save_bandwidth=save)
        assert tuple(a) == ast.literal_eval(b), (kind, save)
    assert ts.HALF_NORM_EXPECTED_VAL == ast.literal_eval(g['half_norm_expected_val'])


def test_pipeline_chunk_schedule_covers_every_read_once():
    """host-only part of tb2_resquiggle_batch: the chunk schedule (no device needed)"""
    import numpy as np
    from tombo_b200 import _lib
    lib = _lib.load()
    fn = lib.tb2_pipeline_chunks
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_int, ctypes.c_int64, ctypes.POINTER(ctypes.c_int64), ctypes.c_int]
    buf = (ctypes.c_int64 * 4096)()
    sm = 148
    unit = sm * 32
    for n in [0, 1, unit, 6 * unit, 6 * unit + 1, 39122, 100000, 1000003]:
        k = fn(sm, n, buf, 4096)
        assert k >= 1, (n, k)
        starts = np.array(buf[:k + 1])
        assert starts[0] == 0 and starts[-1] == n
        sizes = np.diff(starts)
        if n > 0:
            assert np.all(sizes > 0)
        assert np.all(sizes <= 8 * unit) or k == 1
        if n <= 6 * unit:
            assert k == 1                     # small batches are not pipelined
        else:
            assert k >= 2 and sizes[0] == 2 * unit   # short first chunk: its upload is exposed
    assert fn(sm, 10 ** 9, buf, 8) < 0        # capacity is reported, not overrun
    assert fn(sm, -1, buf, 8) < 0
