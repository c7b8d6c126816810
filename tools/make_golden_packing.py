#!/usr/bin/env python
"""Golden vectors for packed language-model batches (fixed-length blocks with per-document position_ids, labels,
seq_idx and cu_seq_lens), recorded from transformers' DataCollatorWithFlattening (its version is stored as `pins`):
python tools/make_golden_packing.py -> tests/golden/packing_hf.json.gz.

The rows are the golden rows' ids: `ids_bpe24k` without eos, `ids_spm24k` without eos and with eos 2 (65 of those rows
are empty).  They come in 8 seeded batches of 64 rows and one batch of the longest row (3558 BPE ids) with the rows
whose SentencePiece ids are empty.  Every batch is packed with block sizes 1 .. 4096 in one call and as a chain of 3
calls at seeded row cuts, each call taking the previous one's rest as its carry.  The pieces come from the rule in
tools/pack_oracle.py; the script asserts that they reassemble into `group_texts`' blocks and that the chain gives the
same blocks as the one call.  Per call it stores N, the piece lengths (the differences of cu_seq_lens), max_length,
the rest's fragment lengths and the CRC32 of every array DataCollatorWithFlattening(return_flash_attn_kwargs=True,
return_seq_idx=True) returns for the pieces; two calls are stored verbatim."""
import gzip
import json
import os
import random
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import pack_oracle as O  # noqa: E402

SEED = 20261021
BATCH = 64
N_BATCHES = 8
BLOCK_SIZES = [1, 2, 3, 8, 17, 64, 128, 512, 4096]
SOURCES = [('bpe24k', 'ids_bpe24k', None), ('spm24k', 'ids_spm24k', None), ('spm24k_eos', 'ids_spm24k', 2)]
VERBATIM = [('bpe24k', 0, 17, 'one'), ('spm24k_eos', 8, 64, 'chain')]
KEYS = ('input_ids', 'labels', 'position_ids', 'seq_idx')


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


def collate(pieces):
    """what the installed collator returns for the pieces, as numpy arrays / ints"""
    from transformers import DataCollatorWithFlattening
    if not pieces:
        return {'input_ids': np.zeros((1, 0), np.int64), 'labels': np.zeros((1, 0), np.int64),
                'position_ids': np.zeros((1, 0), np.int64), 'seq_idx': np.zeros((1, 0), np.int32),
                'cu_seq_lens_q': np.zeros(1, np.int32), 'cu_seq_lens_k': np.zeros(1, np.int32), 'max_length_q': 0,
                'max_length_k': 0}
    c = DataCollatorWithFlattening(return_flash_attn_kwargs=True, return_seq_idx=True)
    return c([{'input_ids': p} for p in pieces], return_tensors='np')


def record(pieces, rest, L, verbatim=False):
    out = collate(pieces)
    flat = O.flatten(pieces)
    for k in KEYS:
        assert out[k].tolist() == [flat[k]], k
        assert out[k].dtype == (np.int32 if k == 'seq_idx' else np.int64), k
    assert out['cu_seq_lens_q'].tolist() == out['cu_seq_lens_k'].tolist() == flat['cu_seq_lens']
    assert out['cu_seq_lens_q'].dtype == np.int32 and out['max_length_q'] == out['max_length_k'] == flat['max_length']
    NL = sum(len(p) for p in pieces)
    assert NL % L == 0
    cu = flat['cu_seq_lens']
    rec = {'N': NL // L, 'pieces': [b - a for a, b in zip(cu, cu[1:])], 'max_length': flat['max_length'],
           'rest': [b - a for a, b in zip(rest[1], rest[1][1:])], 'rest_crc': crc(np.asarray(rest[0], np.int32)),
           'crc': {k: crc(out[k]) for k in KEYS + ('cu_seq_lens_q',)}}
    if verbatim:
        rec['verbatim'] = {k: (v.tolist() if hasattr(v, 'tolist') else v) for k, v in out.items()}
        rec['verbatim_rest'] = [list(rest[0]), list(rest[1])]
    return rec


def main():
    import transformers
    with gzip.open(os.path.join(ROOT, 'tests', 'golden', 'reference_vectors.json.gz'), 'rb') as f:
        rows = json.loads(f.read().decode('utf-8'))['rows']
    rng = random.Random(SEED)
    batches = [sorted(rng.sample(range(len(rows)), BATCH)) for _ in range(N_BATCHES)]
    longest = max(range(len(rows)), key=lambda i: len(rows[i]['ids_bpe24k']))
    batches.append([longest] + [i for i, r in enumerate(rows) if not r['ids_spm24k']])
    cuts = []
    for b in batches:
        c1, c2 = sorted(rng.randint(0, len(b)) for _ in range(2))
        cuts.append([c1, c2])
    out = {'pins': {'transformers': transformers.__version__}, 'seed': SEED, 'batches': batches, 'cuts': cuts,
           'block_sizes': BLOCK_SIZES, 'sources': {}}
    for name, key, eos in SOURCES:
        src = {'key': key, 'eos': eos, 'one': [], 'chain': []}
        for bi, b in enumerate(batches):
            ids = [rows[i][key] for i in b]
            one_b, chain_b = {}, {}
            for L in BLOCK_SIZES:
                verb = [v[3] for v in VERBATIM if v[0] == name and v[1] == bi and v[2] == L]
                pieces, rest = O.pack(ids, L, eos)
                S, _ = O.stream(ids, eos)
                assert O.group_texts(S, L) == O.group_texts([x for p in pieces for x in p], L)
                assert [x for p in pieces for x in p] == S[:len(S) // L * L] and rest[0] == S[len(S) // L * L:]
                one_b[str(L)] = record(pieces, rest, L, 'one' in verb)
                c1, c2 = cuts[bi]
                carry, recs, chained = None, [], []
                for part in (ids[:c1], ids[c1:c2], ids[c2:]):
                    pieces_k, carry_next = O.pack(part, L, eos, carry)
                    recs.append(record(pieces_k, carry_next, L, 'chain' in verb))
                    chained += pieces_k
                    carry = carry_next
                assert chained == pieces and carry == rest
                chain_b[str(L)] = recs
            src['one'].append(one_b)
            src['chain'].append(chain_b)
        out['sources'][name] = src
    path = os.path.join(ROOT, 'tests', 'golden', 'packing_hf.json.gz')
    with gzip.GzipFile(path, 'wb', mtime=0) as f:
        f.write(json.dumps(out, separators=(',', ':')).encode('utf-8'))
    print('wrote %s (%d bytes)' % (path, os.path.getsize(path)))


if __name__ == '__main__':
    main()
