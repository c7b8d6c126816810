"""Drop-in for the reference's `akshar.normalize` (src/akshar/normalize.py), computed by the CUDA normalize kernel.

Same names, arguments and results as the reference; every call -- single string or batch -- runs on the GPU through
libakshar_b200.so (there is no CPU path).  The `*_batch` functions are the new batch entry points: list[str] (or a
device `TextBatch`) in, list[str] (or `TextBatch` with `as_device=True`) out.
"""
from . import _lib as C
from .batch import engine

_STAGE_FLAGS = {
    'normalize_unicode': 0,                                   # normalize.py:13-18
    'semantic_normalize': C.NORM_ROMAN | C.NORM_NO_NFC,       # normalize.py:21-45
    'remove_elongations': C.NORM_COLLAPSE | C.NORM_NO_NFC,    # normalize.py:48-56
    'filter_garbage': C.NORM_FILTER | C.NORM_NO_NFC,          # normalize.py:92-107
    'normalize_hinglish': C.NORM_CLEAN | C.NORM_NO_NFC,       # normalize.py:110-114
}


def _run_flags(batch, flags, as_device=False, device=0):
    tb = engine(device)._normalize(batch, flags)
    return tb if as_device else tb.to_strings()


def _norm_flags(normalize_roman, clean_hinglish):
    return (C.NORM_ROMAN if normalize_roman else 0) | (C.NORM_CLEAN if clean_hinglish else 0)


# ---- batch entry points (new) -----------------------------------------------------------------------
def normalize_batch(texts, normalize_roman=True, clean_hinglish=True, as_device=False, device=0):
    """normalize_text over a batch of sentences"""
    return _run_flags(texts, _norm_flags(normalize_roman, clean_hinglish), as_device, device)


def stage_batch(name, texts, as_device=False, device=0):
    """one of the stand-alone stages (normalize_unicode, semantic_normalize, ...) over a batch"""
    return _run_flags(texts, _STAGE_FLAGS[name], as_device, device)


def roman_phonetic_signature_batch(words, as_device=False, device=0):
    tb = engine(device).signature_batch(words)
    return tb if as_device else tb.to_strings()


# ---- reference API (same signatures) ------------------------------------------------------------------
def normalize_unicode(text):
    return _run_flags([text], _STAGE_FLAGS['normalize_unicode'])[0]


def semantic_normalize(text):
    return _run_flags([text], _STAGE_FLAGS['semantic_normalize'])[0]


def remove_elongations(text):
    return _run_flags([text], _STAGE_FLAGS['remove_elongations'])[0]


def roman_phonetic_signature(word):
    return roman_phonetic_signature_batch([word])[0]


def filter_garbage(text):
    return _run_flags([text], _STAGE_FLAGS['filter_garbage'])[0]


def normalize_hinglish(text):
    return _run_flags([text], _STAGE_FLAGS['normalize_hinglish'])[0]


def normalize_text(text, normalize_roman=True, clean_hinglish=True):
    return _run_flags([text], _norm_flags(normalize_roman, clean_hinglish))[0]
