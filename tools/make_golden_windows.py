#!/usr/bin/env python
"""Golden vectors for the model-ready windows (truncation, stride windows, padding), recorded from HF `tokenizers`
(its version is stored as `pins`):  python tools/make_golden_windows.py -> tests/golden/windows_hf.json.gz.

Three BPE variants (bpe24k.json, bpe_corpus.json, bpe24k.json without its post-processor) encode the golden rows'
`norm` strings in batches of 64 consecutive rows.  Per truncation configuration, every window HF returns (the encoding
and its `overflowing`, in that order) is stored as (start, length) in the row's untruncated content (the row's ids
without template ids, which reference_vectors.json.gz holds); the script asserts that HF's ids are exactly
[bos] + that slice + [eos].  Per padding configuration it stores HF's padded width of every batch and asserts that HF's
padded ids / attention mask are the layout of tools/windows_oracle.py; two batches are also kept verbatim."""
import gzip
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
MODELS = os.path.join(ROOT, 'tests', 'golden', 'models')
BATCH = 64
# (max_length, stride, direction); 's+1' = the template ids + 1, None = truncation off
TRUNC = [(None, 0, 'right'), ('s+1', 0, 'right'), (8, 5, 'left'), (8, 0, 'right'), (32, 7, 'right'), (32, 0, 'left'),
         (128, 31, 'left'), (128, 0, 'right'), (512, 127, 'right'), (512, 0, 'left')]
PAD = [(mode, side, mult) for mode in ('longest', 'max_length') for side in ('right', 'left') for mult in (None, 8)]
VARIANTS = [('bpe24k', 'bpe24k.json', True, 'ids_bpe24k'), ('bpe_corpus', 'bpe_corpus.json', True, 'ids_bpe_corpus'),
            ('bpe24k_no_template', 'bpe24k.json', False, 'ids_bpe24k')]
VERBATIM = [(2, 0, ('longest', 'left', 8)), (6, 73, ('max_length', 'right', None))]    # (TRUNC index, batch, PAD entry)


def trunc_name(t):
    return 'none' if t[0] is None else '%s,%d,%s' % t


def pad_name(p):
    return '%s,%s,%s' % (p[0], p[1], p[2] or 0)


def locate(c, inner, prev, left):
    """position of window `inner` in content c: the first match after the previous window's start (right truncation) or
    the last one ending before the previous window's stop (left)"""
    n, k = len(c), len(inner)
    cands = range(prev[0] + 1 if prev else 0, n - k + 1) if not left else range((prev[1] - 1 if prev else n) - k, -1, -1)
    for a in cands:
        if c[a:a + k] == inner:
            return a
    raise AssertionError('HF window is not a slice of the row content')


def main():
    import tokenizers
    from windows_oracle import windows
    with gzip.open(os.path.join(ROOT, 'tests', 'golden', 'reference_vectors.json.gz'), 'rb') as f:
        rows = json.loads(f.read().decode('utf-8'))['rows']
    norm = [r['norm'] for r in rows]
    batches = [(b, min(b + BATCH, len(rows))) for b in range(0, len(rows), BATCH)]
    out = {'pins': {'tokenizers': tokenizers.__version__}, 'batch': BATCH, 'trunc': [trunc_name(t) for t in TRUNC],
           'pad': [pad_name(p) for p in PAD], 'variants': {}}
    for name, fname, template, key in VARIANTS:
        tk = tokenizers.Tokenizer.from_file(os.path.join(MODELS, fname))
        if not template:
            tk.post_processor = None
        bos, eos = (2, 3) if template else (None, None)
        s = 2 if template else 0
        content = [r[key][1:-1] for r in rows]
        tk.no_truncation()
        tk.no_padding()
        assert [e.ids for e in tk.encode_batch(norm)] == [([bos] if template else []) + c + ([eos] if template else [])
                                                          for c in content]
        V = {'template': template, 'bos': bos, 'eos': eos, 'pad_id': 0, 'windows': {}, 'width': {}, 'verbatim': []}
        for ti, t in enumerate(TRUNC):
            ml = s + 1 if t[0] == 's+1' else t[0]
            left = t[2] == 'left'
            tk.no_padding()
            if ml is None:
                tk.no_truncation()
            else:
                tk.enable_truncation(ml, stride=t[1], direction=t[2])
            spans = []                 # per row: [start0, len0, start1, len1, ...]
            for b0, b1 in batches:
                for r, e in zip(range(b0, b1), tk.encode_batch(norm[b0:b1])):
                    flat, prev = [], None
                    for w in [e] + list(e.overflowing):
                        ids = w.ids
                        assert ids[:1] == [bos] and ids[-1:] == [eos] if template else True
                        inner = ids[1:-1] if template else ids
                        a = locate(content[r], inner, prev, left)
                        prev = (a, a + len(inner))
                        flat += [a, len(inner)]
                    spans.append(flat)
            V['windows'][trunc_name(t)] = spans
            widths = {}
            for p in PAD:
                if p[0] == 'max_length' and ml is None:
                    continue
                tk.enable_padding(direction=p[1], pad_id=0, pad_token='<pad>', length=ml if p[0] == 'max_length' else None,
                                  pad_to_multiple_of=p[2])
                ws = []
                for bi, (b0, b1) in enumerate(batches):
                    encs = tk.encode_batch(norm[b0:b1])
                    hf_ids = [w.ids for e in encs for w in [e] + list(e.overflowing)]
                    hf_mask = [w.attention_mask for e in encs for w in [e] + list(e.overflowing)]
                    o_ids, o_mask, _ = windows([rows[r][key] if template else rows[r][key][1:-1] for r in range(b0, b1)], bos,
                                               eos, ml, t[1], left, True, p[0], p[2], p[1] == 'left', 0, truncate=ml is not None)
                    assert hf_ids == o_ids and hf_mask == o_mask, (name, t, p, bi)
                    ws.append(len(hf_ids[0]))
                    if name == 'bpe24k' and (ti, bi, p) in VERBATIM:
                        V['verbatim'].append({'trunc': trunc_name(t), 'pad': pad_name(p), 'batch': bi, 'input_ids': hf_ids,
                                              'attention_mask': hf_mask})
                widths[pad_name(p)] = ws
            V['width'][trunc_name(t)] = widths
            print(name, trunc_name(t), 'windows', sum(len(x) // 2 for x in spans), flush=True)
        out['variants'][name] = V
    path = os.path.join(ROOT, 'tests', 'golden', 'windows_hf.json.gz')
    with gzip.GzipFile(path, 'wb', mtime=0) as f:
        f.write(json.dumps(out, separators=(',', ':')).encode('utf-8'))
    print('wrote', path, os.path.getsize(path))


if __name__ == '__main__':
    main()
