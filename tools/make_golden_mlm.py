#!/usr/bin/env python
"""Golden vectors for masked language-model batches, recorded from transformers' DataCollatorForLanguageModeling
(its version is stored as `pins`): python tools/make_golden_mlm.py -> tests/golden/mlm_hf.json.gz.

The collator's own `torch_mask_tokens` runs with torch.bernoulli / torch.randint replaced by the Philox draws of
tools/mlm_oracle.py: bernoulli call k draws position (n, j) iff word k of its block, over 2^32, is below the float32
probability the collator passed, and randint returns r_id V >> 32.  The script asserts the collator's call sequence:
three bernoulli calls then randint, or two bernoulli calls when it returns early (m = 1 or r = 0).

Inputs, from a seeded sample of 512 golden rows and the longest one (3558 BPE ids):
  * windows_bpe24k: their `ids_bpe24k` as windows of tools/windows_oracle.py (max_length 128, stride 32, overflowing
    windows, padded with <pad> to the longest);
  * packed_{bpe24k,spm24k}_{256,512}: their `ids_bpe24k` (no eos) / `ids_spm24k` (eos 2) as the packed blocks of
    tools/pack_oracle.py.
Tokenizers: bpe24k.json as PreTrainedTokenizerFast with <pad> <unk> <s> </s> <mask> declared; spm24k.model as a
`tokenizers` Unigram of its (piece, score) list (unk_id 0, byte_fallback) with <unk> <s> </s> <mask> declared.
Per input, setting (p, m, r) and key (seed, epoch, row_base) it stores the counts of selected / replaced / random
positions and the CRC32 of the int64 input_ids and labels the collator returned; two calls are stored verbatim."""
import gzip
import json
import os
import random
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import mlm_oracle as O  # noqa: E402
import pack_oracle as P  # noqa: E402
import windows_oracle as W  # noqa: E402

SEED = 20261022
N_ROWS = 512
SETTINGS = [(.15, .8, .1), (.3, .8, .1), (.15, 1, 0), (.5, 0, 1), (0, .8, .1), (1, .8, .1), (.4, .5, .5), (.2, .7, 0)]
KEYS = [(0, 0, 0), (2 ** 64 - 1, 2 ** 32 - 1, 2 ** 32 - 3), (987654321, 7, 2 ** 40)]
WINDOWS = dict(max_length=128, stride=32, pad_id=0)
# (input, rows [a, b), setting, key) of the calls stored verbatim
VERBATIM = [('windows_bpe24k', (0, 4), 0, 0), ('packed_spm24k_512', (0, 2), 3, 1)]


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a, np.int64).tobytes())


def tokenizers():
    from tokenizers import Tokenizer
    from tokenizers.models import Unigram
    from transformers import PreTrainedTokenizerFast
    import sentencepiece as spm
    models = os.path.join(ROOT, 'tests', 'golden', 'models')
    bpe = PreTrainedTokenizerFast(tokenizer_file=os.path.join(models, 'bpe24k.json'), pad_token='<pad>', unk_token='<unk>',
                                  bos_token='<s>', eos_token='</s>', mask_token='<mask>')
    sp = spm.SentencePieceProcessor(model_file=os.path.join(models, 'spm24k.model'))
    vocab = [(sp.id_to_piece(i), sp.get_score(i)) for i in range(sp.get_piece_size())]
    uni = PreTrainedTokenizerFast(tokenizer_object=Tokenizer(Unigram(vocab, unk_id=0, byte_fallback=True)), unk_token='<unk>',
                                  bos_token='<s>', eos_token='</s>', mask_token='<mask>')
    return {'bpe24k': bpe, 'spm24k': uni}


def collate(tok, ids, p, m, r, seed, epoch, row_base):
    """the collator's torch_mask_tokens on ids (int64 [N, L]) with the Philox draws -> (input_ids, labels, counts)"""
    import torch
    from transformers import DataCollatorForLanguageModeling
    c = DataCollatorForLanguageModeling(tokenizer=tok, mlm=True, mlm_probability=p, mask_replace_prob=m, random_replace_prob=r)
    N, L = ids.shape
    U = O.draws(N, L, seed, epoch, row_base)
    V = len(tok)
    calls, drawn = [], []
    real = torch.bernoulli, torch.randint

    def bernoulli(prob, generator=None):
        k = len(calls)
        assert calls == ['b'] * k and k < 3 and prob.dtype == torch.float32 and tuple(prob.shape) == (N, L)
        calls.append('b')
        out = (torch.from_numpy(U[k].astype(np.float64)) / 2 ** 32 < prob.double()).to(prob.dtype)
        drawn.append(out.bool().numpy())
        return out

    def randint(high, size, dtype=None, generator=None):
        assert calls == ['b'] * 3 and high == V and tuple(size) == (N, L) and dtype == torch.long
        calls.append('r')
        return torch.from_numpy(((U[3].astype(np.uint64) * np.uint64(V)) >> np.uint64(32)).astype(np.int64))
    torch.bernoulli, torch.randint = bernoulli, randint
    try:
        inputs, labels = c.torch_mask_tokens(torch.from_numpy(ids.copy()))
    finally:
        torch.bernoulli, torch.randint = real
    early = m == 1 or r == 0
    assert calls == (['b', 'b'] if early else ['b', 'b', 'b', 'r']), calls
    inputs, labels = inputs.numpy(), labels.numpy()
    sel = labels != -100
    rep = drawn[1] & sel
    rnd = np.zeros_like(sel) if early else drawn[2] & sel & ~rep
    return inputs, labels, [int(sel.sum()), int(rep.sum()), int(rnd.sum())]


def inputs(rows):
    """name -> (model, int64 [N, L] input_ids, pad_id, description)"""
    out = {}
    bpe = [r['ids_bpe24k'] for r in rows]
    ids, _, _ = W.windows(bpe, 2, 3, WINDOWS['max_length'], WINDOWS['stride'], False, True, 'longest', None, False, WINDOWS['pad_id'])
    out['windows_bpe24k'] = ('bpe24k', np.asarray(ids, np.int64), WINDOWS['pad_id'], dict(kind='windows', **WINDOWS))
    for model, key, eos in (('bpe24k', 'ids_bpe24k', None), ('spm24k', 'ids_spm24k', 2)):
        for L in (256, 512):
            pieces, _ = P.pack([r[key] for r in rows], L, eos)
            flat = P.flatten(pieces)['input_ids']
            out['packed_%s_%d' % (model, L)] = (model, np.asarray(flat, np.int64).reshape(-1, L), None,
                                                dict(kind='packed', block_size=L, eos_id=eos))
    return out


def main():
    import transformers
    with gzip.open(os.path.join(ROOT, 'tests', 'golden', 'reference_vectors.json.gz'), 'rb') as f:
        all_rows = json.loads(f.read().decode('utf-8'))['rows']
    longest = max(range(len(all_rows)), key=lambda i: len(all_rows[i]['ids_bpe24k']))
    sample = sorted(set(random.Random(SEED).sample(range(len(all_rows)), N_ROWS)) | {longest})
    rows = [all_rows[i] for i in sample]
    toks = tokenizers()
    models = {}
    for name, tok in toks.items():
        models[name] = {'V': len(tok), 'mask_id': tok.mask_token_id, 'special': sorted(tok.all_special_ids)}
    assert models['bpe24k'] == {'V': 24000, 'mask_id': 4, 'special': [0, 1, 2, 3, 4]}, models
    assert models['spm24k'] == {'V': 24000, 'mask_id': 3, 'special': [0, 1, 2, 3]}, models
    out = {'pins': {'transformers': transformers.__version__}, 'seed': SEED, 'rows': sample, 'settings': SETTINGS, 'keys': KEYS,
           'models': models, 'inputs': {}, 'calls': {}, 'verbatim': []}
    for name, (model, ids, pad, desc) in inputs(rows).items():
        out['inputs'][name] = dict(desc, model=model, pad_id=pad, shape=list(ids.shape), crc=crc(ids))
        recs = []
        for p, m, r in SETTINGS:
            per_key = []
            for seed, epoch, row_base in KEYS:
                got, labels, counts = collate(toks[model], ids, p, m, r, seed, epoch, row_base)
                want = O.mask(ids, models[model]['special'], models[model]['V'], models[model]['mask_id'], seed, p, m, r, epoch,
                              row_base, pad)
                assert np.array_equal(got, want[0]) and np.array_equal(labels, want[1]) and tuple(counts) == want[2], (name, p, m, r)
                per_key.append({'counts': counts, 'crc': {'input_ids': crc(got), 'labels': crc(labels)}})
            recs.append(per_key)
        out['calls'][name] = recs
        for vname, (a, b), si, ki in VERBATIM:
            if vname != name:
                continue
            seed, epoch, row_base = KEYS[ki]
            got, labels, _ = collate(toks[model], ids[a:b], *SETTINGS[si], seed, epoch, row_base + a)
            out['verbatim'].append({'input': name, 'rows': [a, b], 'setting': si, 'key': ki, 'input_ids': got.tolist(),
                                    'labels': labels.tolist()})
    path = os.path.join(ROOT, 'tests', 'golden', 'mlm_hf.json.gz')
    with gzip.GzipFile(path, 'wb', mtime=0) as f:
        f.write(json.dumps(out, separators=(',', ':')).encode('utf-8'))
    print('wrote %s (%d bytes)' % (path, os.path.getsize(path)))


if __name__ == '__main__':
    main()
