#!/usr/bin/env python
"""Golden vectors for the wide-Unicode fuzz tests, recorded from the libraries the reference calls (unicodedata NFC,
regex \\X, tokenizers, sentencepiece; their versions are stored as `pins`):  python tools/make_golden_fuzz.py
-> tests/golden/library_fuzz.json.gz.  The rows come from the generators of the tests that read the file."""
import gzip
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'oracle'), os.path.join(ROOT, 'tools'), os.path.join(ROOT, 'tests')):
    sys.path.insert(0, p)
MODELS = os.path.join(ROOT, 'tests', 'golden', 'models')


def main():
    import unicodedata
    import regex
    import sentencepiece
    import tokenizers
    from test_span_walkers import wide_unicode_lines
    from test_subword_cores import wide_unicode_encoder_lines
    pins = {'regex': regex.__version__, 'tokenizers': tokenizers.__version__, 'sentencepiece': sentencepiece.__version__,
            'unicodedata': unicodedata.unidata_version}
    rows = wide_unicode_lines()
    walkers = {'rows': rows, 'nfc': [unicodedata.normalize('NFC', s) for s in rows],
               'clusters': [regex.findall(r'\X', s) for s in rows]}
    norm = wide_unicode_encoder_lines()
    tk = tokenizers.Tokenizer.from_file(os.path.join(MODELS, 'bpe24k.json'))
    sp = sentencepiece.SentencePieceProcessor()
    sp.Load(os.path.join(MODELS, 'spm24k.model'))
    encoders = {'rows': norm, 'bpe24k': [tk.encode(s).ids for s in norm], 'spm24k': [sp.EncodeAsIds(s) for s in norm]}
    path = os.path.join(ROOT, 'tests', 'golden', 'library_fuzz.json.gz')
    with gzip.GzipFile(path, 'wb', mtime=0) as f:
        f.write(json.dumps({'pins': pins, 'walkers': walkers, 'encoders': encoders}, ensure_ascii=False,
                           separators=(',', ':')).encode('utf-8'))
    print('wrote', path, os.path.getsize(path))


if __name__ == '__main__':
    main()
