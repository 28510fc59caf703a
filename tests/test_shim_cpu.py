"""CPU: host-side pieces of the Python mirror API -- batch packing (one bad read never
aborts a batch), error typing, and the two helpers re-expressed in vectorised form checked
against the unmodified reference on random inputs (digests of its outputs recorded by
tests/golden/make_reference_api_golden.py)."""
import numpy as np
import pytest

import golden_util as gu


def _map_res(raw, seq):
    from tombo_b200 import tombo_helper as th
    return th.resquiggleResults(
        align_info=th.alignInfo('r', 'BaseCalled_template', 0, 0, 0, 0, len(seq), 0),
        genome_loc=th.genomeLocation(0, '+', 'chr'), genome_seq=seq, mean_q_score=10.0,
        raw_signal=raw)


def test_pack_reads_keeps_a_read_without_signal_as_an_empty_slice():
    from tombo_b200 import resquiggle as rq
    reads = [_map_res(np.arange(10, dtype=np.float64), 'ACGTACGTAC'),
             _map_res(None, 'ACGTACGT'),
             _map_res(np.arange(7, dtype=np.float64), 'ACGTACG')]
    raw, raw_off, seq, seq_off = rq.pack_reads(reads)
    assert raw_off.tolist() == [0, 10, 10, 17]          # the None read owns no samples
    assert seq_off.tolist() == [0, 10, 18, 25]
    assert raw.shape[0] == 17 and raw.dtype == np.float64
    # all-int16 batches stay int16 (the DAC dtype), a None read does not break that
    reads = [_map_res(np.arange(5, dtype=np.int16), 'ACGTA'), _map_res(None, 'ACGTA')]
    raw, raw_off, _, _ = rq.pack_reads(reads)
    assert raw.dtype == np.int16 and raw_off.tolist() == [0, 5, 5]


def test_status_exception_types_follow_the_reference_buckets():
    from tombo_b200 import resquiggle as rq, tombo_helper as th
    assert isinstance(rq._status_exception(17), th.TomboError)          # no raw signal
    assert str(rq._status_exception(17)).startswith('Must have raw signal')
    for st in (100, 200, 202):       # UNEXPECTED / CUDA / CAPACITY: not Tombo errors
        e = rq._status_exception(st)
        assert isinstance(e, rq.LibraryError) and not isinstance(e, th.TomboError)


def test_batcher_files_library_errors_as_non_tombo():
    from tombo_b200 import resquiggle as rq, tombo_helper as th, worker

    def fake(map_results, *a, **k):
        return [rq._status_exception(100), rq._status_exception(17), map_results[2]]
    b = worker.ReadBatcher(None, None, resquiggle_fn=fake)
    for i in range(3):
        b.add(_map_res(np.zeros(4), 'ACGT'), 'f%d' % i)
    out = b.flush()
    assert out[0][1][0] is True and out[0][1][1][2] is False      # 'Unexpected error' bucket
    assert out[1][1][0] is True and out[1][1][1][2] is True       # TomboError bucket
    assert out[2][1][0] is False


def test_trim_seq_and_means_equals_reference_on_random_regions():
    from tombo_b200 import tombo_stats as ts, tombo_helper as th
    g = gu.load('reference_api')
    ok, dig = g['trim_ok'], g['trim_digest']
    assert ok.shape[0] == dig.shape[0] == 3000
    for it, (seq, means, args) in enumerate(gu.trim_cases()):
        b = gu.trim_result(ts.trim_seq_and_means, th.TomboError, seq, means, args)
        assert (b[0] == 'ok') == bool(ok[it]), (it, args, b)
        assert np.array_equal(gu.digest(b), dig[it]), (it, args, b)
    assert ok.sum() > 500 and (~ok).sum() > 500


def test_remove_stall_cpts_equals_reference():
    from tombo_b200 import resquiggle as rq
    dig = gu.load('reference_api')['stall_digest']
    assert dig.shape[0] == 1000
    for it, (ints, cp) in enumerate(gu.stall_cases()):
        b = np.asarray(rq._remove_stall_cpts(ints, cp), dtype=np.int64).tolist()
        assert np.array_equal(gu.digest(b), dig[it]), (it, ints)


def test_write_new_fast5_group_opens_path_likes_and_always_closes(monkeypatch, tmp_path):
    """bytes / pathlib paths are opened (the reference opens anything that is not an open
    file), and the file is closed even when the write raises"""
    import sys
    import types
    from tombo_b200 import tombo_helper as th
    opened = []

    class FakeFile(object):
        def __init__(self, fn, mode):
            opened.append(self); self.fn = fn; self.closed = False

        def __getitem__(self, k):
            raise KeyError(k)          # make the write fail

        def close(self):
            self.closed = True
    monkeypatch.setitem(sys.modules, 'h5py', types.SimpleNamespace(File=FakeFile))
    res = _map_res(np.zeros(8), 'ACG')._replace(
        segs=np.array([0, 2, 5, 8]), scale_values=th.scaleValues(0.0, 1.0, -5.0, 5.0, 5.0))
    for target in (tmp_path / 'x.fast5', str(tmp_path / 'y.fast5').encode()):
        with pytest.raises(th.TomboError, match='Error writing resquiggle information'):
            th.write_new_fast5_group(target, 'RawGenomeCorrected_000', res, 'median', False,
                                     norm_means=np.zeros(3))
        assert opened[-1].closed and isinstance(opened[-1].fn, str)
    # failures while building the Events table surface as the reference's message
    with pytest.raises(th.TomboError, match='Error computing new events'):
        th.write_new_fast5_group(FakeFile('z', 'r+'), 'g', res._replace(genome_seq='ACé'),
                                 'median', False, norm_means=np.zeros(3))
