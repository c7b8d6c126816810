import gzip
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'oracle'), os.path.join(ROOT, 'tools')):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
MODELS = os.path.join(GOLDEN, 'models')

# the reference's own test files kept as fixtures: run (unmodified) by test_gpu_parity.py, never collected directly
collect_ignore_glob = ['golden/ref_tests/*']


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


@pytest.fixture(scope='session')
def golden():
    with gzip.open(os.path.join(GOLDEN, 'reference_vectors.json.gz'), 'rb') as f:
        return json.loads(f.read().decode('utf-8'))


@pytest.fixture(scope='session')
def decode_fuzz():
    """id rows decoded / detokenized by the unmodified reference (tools/make_golden_decode.py)"""
    with gzip.open(os.path.join(GOLDEN, 'decode_fuzz.json.gz'), 'rb') as f:
        return json.loads(f.read().decode('utf-8'))


@pytest.fixture(scope='session')
def models_dir():
    return MODELS


@pytest.fixture(scope='session')
def bpe_rows(golden):
    """the golden rows the BPE path is checked on: all of them (until round 2 the rows with a code point HF's NFKC treats
    differently from NFC -- U+09FE, newer than HF's Unicode tables -- had to be left out)"""
    return golden['rows']


@pytest.fixture(scope='session')
def golden_raw():
    """vectors recorded from the unmodified reference with clean_hinglish=False (tools/make_golden_raw.py)"""
    with gzip.open(os.path.join(GOLDEN, 'reference_vectors_raw.json.gz'), 'rb') as f:
        return json.loads(f.read().decode('utf-8'))


@pytest.fixture(scope='session')
def library_fuzz():
    """what the libraries the reference calls (unicodedata, regex, tokenizers, sentencepiece) returned for the wide-Unicode
    fuzz rows (tools/make_golden_fuzz.py)"""
    with gzip.open(os.path.join(GOLDEN, 'library_fuzz.json.gz'), 'rb') as f:
        return json.loads(f.read().decode('utf-8'))
