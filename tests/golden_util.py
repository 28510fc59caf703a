"""Helpers to replay tests/golden/*.npz (outputs of the unmodified reference)."""
import hashlib
import os

import numpy as np

from tombo_b200 import synthetic as syn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
READ_CONFIGS = ['dna_static4k', 'dna_adapt4k', 'dna_adapt_bw400', 'dna_long_subsample',
                'dna_int16_stable', 'dna_rescue', 'rna_8k',
                # round 2: BASELINE.json configs[2..4] shapes
                'dna_c5_bw1200', 'dna_c3_rescue_long', 'rna_const_scale']
RNA_ALN = (6, 4, 500, 1500, 20.0, 50, 1000, 3000, 250)
DNA_SEG, RNA_SEG = (5, 3, 1, 5), (12, 6, 2, 15)


def load(name):
    return np.load(os.path.join(GOLDEN, name + '.npz'), allow_pickle=False)


def reads_of(g):
    kind = str(g['kind'])
    kmer_ref, cpos = syn.make_kmer_ref(kind, 0)
    reads = []
    for i in range(int(g['nreads'])):
        kw = {}
        if bool(g['int16']):
            kw['int16'] = True
        if bool(g['stall']):
            kw['stall'] = (300 + i, 1500)
        if 'stall_at' in g.files and int(g['stall_at'][i, 0]) >= 0:
            kw['stall'] = (int(g['stall_at'][i, 0]), int(g['stall_at'][i, 1]))
        r = syn.make_read(kmer_ref, cpos, int(g['nbases'][i]), int(g['seed0']) + i, kind=kind, **kw)
        assert float(np.sum(np.asarray(r.raw, dtype=np.float64))) == float(g['raw_checksum'][i]), \
            'synthetic generator drifted from the golden inputs'
        reads.append(r)
    return kind, kmer_ref, cpos, reads


def const_scale_of(g):
    if 'const_scale' in g.files and not np.isnan(float(g['const_scale'])):
        return float(g['const_scale'])
    return None


def params_of(g, RP):
    kind = str(g['kind'])
    aln = tuple(g['aln']) if g['aln'].shape[0] else RNA_ALN
    aln = tuple(float(a) if i in (0, 1, 4) else int(a) for i, a in enumerate(aln))
    seg = DNA_SEG if kind == 'DNA' else RNA_SEG
    return RP(aln, seg, rna=(kind == 'RNA')), RP(aln, seg, rna=(kind == 'RNA'), save=True)


def levels(genome_seq, kmer_ref):
    means, sds = syn.kmer_table(kmer_ref)
    k = len(kmer_ref[0][0])
    codes = syn.seq_to_codes(genome_seq).astype(np.int64)
    nb = codes.shape[0] - k + 1
    kidx = np.zeros(nb, dtype=np.int64)
    for j in range(k):
        kidx = kidx * 4 + codes[j:j + nb]
    return means[kidx], sds[kidx]


def expected(g, i):
    s = g['scalars'][i]
    a, b = int(g['seg_off'][i]), int(g['seg_off'][i + 1])
    return dict(message=str(g['messages'][i]), segs=g['segs'][a:b], shift=s[0], scale=s[1],
                lower_lim=s[2], upper_lim=s[3], sig_match_score=s[4],
                read_start_rel_to_raw=int(s[5]) if not np.isnan(s[5]) else None,
                calls=int(s[6]), rescued=bool(s[7]), n_iters=int(s[8]),
                norm_params_changed=bool(s[9]))


def digest(value):
    """16-byte SHA-256 prefix of repr(value): a golden for outputs too large to store whole.
    Callers pass plain Python values (str, int, float, lists, tuples), whose repr is exact."""
    return np.frombuffer(hashlib.sha256(repr(value).encode()).digest()[:16], dtype=np.uint8)


def trim_cases():
    """3000 seeded argument sets for trim_seq_and_means: (seq, means, args)."""
    rs = np.random.RandomState(3)
    for _ in range(3000):
        K = int(rs.choice([5, 6, 7])); cp = int(rs.randint(0, K))
        L = int(rs.randint(K, 40))
        seq = ''.join(rs.choice(list('ACGT'), L + K - 1))
        means = rs.normal(size=L + K - 1)
        args = (int(rs.randint(0, 50)),)
        reg_start = int(rs.randint(0, 60))
        args += (reg_start, reg_start + int(rs.randint(1, 60)), str(rs.choice(['+', '-'])), K, cp,
                 int(rs.randint(0, 4)), int(rs.randint(0, 8)))
        yield seq, means, args


def trim_result(fn, err, seq, means, args):
    """fn(seq, means, *args) as plain values: ('ok', kmers, means, r_start, motif seq) or
    ('err', message) for an exception of type err."""
    try:
        k, mm, r, ms = fn(seq, means.copy(), *args)
        return ('ok', [str(x) for x in k], [float(x) for x in mm], int(r), str(ms))
    except err as e:
        return ('err', str(e))


def stall_cases():
    """1000 seeded (stall intervals, sorted change points) pairs for remove_stall_cpts."""
    rs = np.random.RandomState(4)
    for _ in range(1000):
        ns = int(rs.randint(0, 6))
        ints = np.sort(rs.choice(np.arange(0, 2000), 2 * ns, replace=False)).reshape(-1, 2)
        cp = np.sort(rs.choice(np.arange(0, 2000), int(rs.randint(1, 300)),
                               replace=False)).astype(np.int64)
        yield [tuple(int(v) for v in x) for x in ints], cp
