"""Golden for the Python-side API from the UNMODIFIED reference (oracle/_ref): the default
parameters, the namedtuple layouts, load_resquiggle_parameters and HALF_NORM_EXPECTED_VAL
(reference_api.json, values as repr strings so tuples stay tuples), and digests of
trim_seq_and_means / remove_stall_cpts on the seeded cases of tests/golden_util.py
(reference_api.npz).    python tests/golden/make_reference_api_golden.py"""
import ast
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'oracle'))
sys.path.insert(0, os.path.dirname(HERE))

import golden_util as gu  # noqa: E402

NAMEDTUPLES = ('alignInfo', 'readData', 'scaleValues', 'resquiggleParams', 'resquiggleResults',
               'dpResults', 'genomeLocation', 'seqSampleType', 'stallParams', 'channelInfo')


def plain(v):
    return v.item() if isinstance(v, np.generic) else v


def literal(v):
    r = repr(plain(v))
    assert ast.literal_eval(r) == plain(v), r
    return r


def main():
    import ref_harness as rh
    m = rh.load_reference()
    th, ts = m['th'], m['ts']
    import tombo._default_parameters as rdp
    out = {'default_parameters': {n: literal(getattr(rdp, n)) for n in dir(rdp) if n.isupper()},
           'namedtuple_fields': {nt: list(getattr(th, nt)._fields) for nt in NAMEDTUPLES},
           'half_norm_expected_val': literal(ts.HALF_NORM_EXPECTED_VAL),
           'resquiggle_parameters': []}
    for kind in ('DNA', 'RNA'):
        for save in (False, True):
            p = ts.load_resquiggle_parameters(th.seqSampleType(kind, kind == 'RNA'),
                                              use_save_bandwidth=save)
            out['resquiggle_parameters'].append(
                [kind, save, literal(tuple(plain(v) for v in p))])
    json.dump(out, open(os.path.join(HERE, 'reference_api.json'), 'w'), sort_keys=True, indent=1)

    trim = [gu.trim_result(ts.trim_seq_and_means, th.TomboError, *c) for c in gu.trim_cases()]
    stall = [np.asarray(ts.remove_stall_cpts(ints, cp), dtype=np.int64).tolist()
             for ints, cp in gu.stall_cases()]
    np.savez_compressed(os.path.join(HERE, 'reference_api.npz'),
                        trim_ok=np.array([t[0] == 'ok' for t in trim]),
                        trim_digest=np.stack([gu.digest(t) for t in trim]),
                        stall_digest=np.stack([gu.digest(s) for s in stall]))
    print('written reference_api.json, reference_api.npz')


if __name__ == '__main__':
    main()
