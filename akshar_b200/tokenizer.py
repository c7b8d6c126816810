"""Drop-in for the reference's `akshar.tokenizer.aksharTokenizer` (src/akshar/tokenizer.py) on the CUDA hot path.

Same constructor, attributes, methods, return types and exceptions as the reference; `tokenize_batch` /
`encode_batch` are the new batch entry points and return ragged token-id tensors.  The model files are the ones the
reference's scripts/train_bpe.py (HuggingFace tokenizers JSON) and scripts/train_spm.py (SentencePiece ModelProto)
write; they are parsed by libakshar_b200.so itself, `tokenizers` / `sentencepiece` are not needed at run time.
"""
import os
from typing import List, Optional, Union

from . import _lib as C
from .batch import engine
from .normalize import normalize_text, normalize_batch
from .segment import (segment_akshars, detect_code_switches, analyze_text_composition, segment_akshars_batch,
                      analyze_text_composition_batch, detect_code_switches_batch, normalize_and_segment_batch)

_SPM_NORMAL, _SPM_UNKNOWN, _SPM_CONTROL, _SPM_USER, _SPM_UNUSED, _SPM_BYTE = 1, 2, 3, 4, 5, 6


class _CudaModel:
    """what `self.model` holds: the vocabulary of the model loaded into the device context"""

    def __init__(self, eng, kind):
        self.kind = kind                       # 0 BPE, 1 Unigram
        self.size, self.vocab = eng.vocab(kind)
        self._ids = None

    def token(self, i):
        return self.vocab[i][0]

    def piece_id(self, piece):
        if self._ids is None:
            self._ids = {}
            for i, (p, _) in enumerate(self.vocab):
                if p is not None and p != '':
                    self._ids.setdefault(p, i)
        return self._ids.get(piece)


class aksharTokenizer:
    """reference tokenizer.py:18-288"""

    def __init__(self, model_path: Optional[str] = None, model_type: str = "sentencepiece", normalize_roman: bool = True,
                 clean_hinglish: bool = True, device: int = 0):
        self.model_path = model_path
        self.normalize_roman = normalize_roman
        self.clean_hinglish = clean_hinglish
        self.model = None
        self._configured_model_type = model_type
        self._device = device
        if model_path and os.path.exists(model_path):
            self._load_model()
        else:
            self.model_type = "akshar"        # reference tokenizer.py:69-71: silent fallback

    def _load_model(self):
        model_type = self._configured_model_type
        # one context per tokenizer so that two tokenizers with different models can coexist
        from .batch import Engine
        if model_type == "sentencepiece":
            self._eng = Engine(self._device)
            try:
                self._eng.load_spm(self.model_path)
            except C.AksharCudaError as e:
                raise RuntimeError(str(e))        # SentencePiece raises RuntimeError on an unparsable ModelProto
            self.model = _CudaModel(self._eng, 1)
            self.model_type = "sentencepiece"
        elif model_type == "bpe":
            self._eng = Engine(self._device)
            try:
                self._eng.load_bpe(self.model_path)
            except C.AksharCudaError as e:
                raise Exception(str(e))           # tokenizers raises a bare Exception on a bad JSON
            self.model = _CudaModel(self._eng, 0)
            self.model_type = "bpe"
        else:
            raise ValueError(f"unknown model_type: {model_type}")

    # ------------------------------------------------------------------ reference API
    def preprocess(self, text: str) -> str:
        return normalize_batch([text], self.normalize_roman, self.clean_hinglish, device=self._device)[0]

    def tokenize(self, text: str, return_metadata: bool = False) -> Union[List[str], dict]:
        if self.model is None:
            # normalize + akshars in one library call (two host synchronisations instead of eight)
            norms, aks = normalize_and_segment_batch([text], self.normalize_roman, self.clean_hinglish, device=self._device)
            norm, tokens = norms[0], aks[0]
        else:
            norm = self.preprocess(text)
            tokens = self._pieces(self._encode_normalized([norm])[0])
        if return_metadata:
            meta = analyze_text_composition_batch([norm], device=self._device)[0]
        if return_metadata:
            meta['tokens'] = tokens
            meta['token_count'] = len(tokens)
            meta['original_text'] = text
            meta['normalized_text'] = norm
            return meta
        return tokens

    def encode(self, text: str) -> List[int]:
        norm = self.preprocess(text)
        if self.model is None:
            raise ValueError("need model for IDs")
        return self._encode_normalized([norm])[0]

    def decode(self, ids: List[int]) -> str:
        if self.model is None:
            raise ValueError("need model to decode")
        return self.decode_batch([ids])[0]

    def detokenize(self, tokens: List[str]) -> str:
        """reference tokenizer.py:221-246.  Token strings that are pieces of the loaded model (what `tokenize` returns) are
        joined on the device from their ids; the reference also accepts arbitrary strings, which have no ids: for those
        (and without a model) the joining expression of tokenizer.py:236-246 is evaluated as it stands."""
        if self.model is not None:
            ids = [self.model.piece_id(t) for t in tokens]
            if all(i is not None for i in ids):
                return self.detokenize_batch([ids])[0]
        if self.model_type == "sentencepiece":
            return ''.join(tokens).replace('▁', ' ').strip()
        elif self.model_type == "bpe":
            return ' '.join(tokens).replace(' ##', '').replace('Ġ', ' ').strip()
        return ''.join(tokens)

    def explain(self, text: str) -> dict:
        norm = self.preprocess(text)
        return {
            'original': text,
            'normalized': norm,
            'akshars': segment_akshars_batch([norm], device=self._device)[0],
            'code_switches': detect_code_switches_batch([norm], device=self._device)[0],
            'tokens': self.tokenize(text),
            'stats': analyze_text_composition_batch([norm], device=self._device)[0],
        }

    def vocab_size(self) -> int:
        return 0 if self.model is None else self.model.size

    # ------------------------------------------------------------------ batch API (new)
    def encode_batch(self, texts, as_device=False):
        """encode() over a batch: list[list[int]], or with as_device=True (Ragged int32 ids + int64 row_splits on
        the device, normalized TextBatch).  normalize and encode are enqueued back to back without a host sync."""
        if self.model is None:
            raise ValueError("need model for IDs")
        ids, norm = self._eng.tokenizer_encode_batch(texts, self.model.kind, self.normalize_roman, self.clean_hinglish)
        if as_device:
            return ids, norm
        return [r.tolist() for r in ids.rows()]

    def encode_batch_tensors(self, texts, text_pair=None, **kwargs):
        """encode() over a batch, returned as the dense tensors a model takes: encode_batch(as_device=True) followed by
        Engine.windows_batch with the same keywords (max_length, padding, truncation, stride, return_overflowing_tokens,
        pad_to_multiple_of, padding_side, truncation_side, pad_id) -> dict of int64 device tensors input_ids,
        attention_mask (and overflow_to_sample_mapping), as transformers' tokenizer(texts, ..., return_tensors='pt').
        text_pair: the second texts of sentence pairs, as transformers' tokenizer(texts, text_pair, ...); texts and pairs
        are encoded in one call and windowed through the model's pair template (truncation may then also be
        'longest_first', 'only_first', 'only_second' or 'do_not_truncate')"""
        if self.model is None:
            raise ValueError("need model for IDs")
        if text_pair is None:
            ids, _ = self.encode_batch(texts, as_device=True)
            return self._eng.windows_batch(ids, self.model.kind, **kwargs)
        texts, text_pair = list(texts), list(text_pair)
        if len(texts) != len(text_pair):
            raise ValueError('texts and text_pair must hold the same number of texts')
        ids, _ = self.encode_batch(texts + text_pair, as_device=True)
        n = len(texts)
        return self._eng.windows_batch((ids.values, ids.splits[:n + 1]), self.model.kind,
                                       pair_ids=(ids.values, ids.splits[n:]), **kwargs)

    def encode_batch_packed(self, texts, block_size, **kwargs):
        """encode() over a batch, packed into fixed blocks for causal-LM training: encode_batch(as_device=True) followed by
        Engine.pack_batch with the same keywords (eos_id, carry, separator_id, return_position_ids, return_seq_idx,
        return_flash_attn_kwargs) -> (batch, rest) as pack_batch returns them.  eos_id defaults to None: the rows of a
        BPE model already end in its `</s>`, while SentencePiece rows carry neither `<s>` nor `</s>`, so SentencePiece
        users pass the model's `</s>` id (2 for spm24k.model) to keep the documents of the stream apart."""
        if self.model is None:
            raise ValueError("need model for IDs")
        ids, _ = self.encode_batch(texts, as_device=True)
        return self._eng.pack_batch(ids, block_size, **kwargs)

    def encode_batch_mlm(self, texts, seed, block_size=None, text_pair=None, mlm_probability=0.15, mask_replace_prob=0.8,
                         random_replace_prob=0.1, epoch=0, row_base=0, **kwargs):
        """encode() over a batch, masked for masked-LM training as transformers' run_mlm.py batches it, in one of its two
        modes.  Without block_size: encode_batch_tensors(texts, text_pair, **kwargs) followed by Engine.mlm_mask (the
        window index is the row; the pad id of the windows is special) -> that dict with `labels` added.  With
        block_size: encode_batch_packed(texts, block_size, **kwargs) followed by Engine.mlm_mask (the block index is the
        row) -> (batch, rest) with the causal-LM labels replaced by the masked-LM ones; position_ids, seq_idx and
        cu_seq_lens stay.  seed, the probabilities, epoch and row_base are those of Engine.mlm_mask."""
        if self.model is None:
            raise ValueError("need model for IDs")
        mlm = dict(seed=seed, mlm_probability=mlm_probability, mask_replace_prob=mask_replace_prob,
                   random_replace_prob=random_replace_prob, epoch=epoch, row_base=row_base)
        if block_size is None:
            batch = self.encode_batch_tensors(texts, text_pair, **kwargs)
            pad = kwargs.get('pad_id')
            pad = self._eng.pad_id(self.model.kind) if pad is None else pad
            batch['labels'] = self._eng.mlm_mask(batch['input_ids'], self.model.kind, pad_id=pad, **mlm)[1]
            return batch
        if text_pair is not None:
            raise ValueError('text_pair is not taken with block_size: packed blocks hold single texts')
        batch, rest = self.encode_batch_packed(texts, block_size, **kwargs)
        batch['labels'] = self._eng.mlm_mask(batch['input_ids'], self.model.kind, **mlm)[1]
        return batch, rest

    def encode_batch_host(self, h_data, h_offsets, out_ids=None, out_splits=None, compact=False):
        """encode() over a batch given as pinned host tensors (uint8 text, int64 row offsets) -> pinned host tensors
        (int32 ids, int64 row_splits), or with compact=True a `CompactIds` (uint16 ids, int32 chunk-relative splits: a third
        of the bytes over the host link); copies and kernels are pipelined over three streams.  The results live in buffers
        the engine reuses: see Engine.encode_host_pipelined."""
        if self.model is None:
            raise ValueError("need model for IDs")
        return self._eng.encode_host_pipelined(h_data, h_offsets, self.model.kind, self.normalize_roman, self.clean_hinglish,
                                               out_ids=out_ids, out_splits=out_splits, compact=compact)

    def _ids_to_text(self, rows, form):
        import torch
        if isinstance(rows, tuple):                       # (ids tensor, splits tensor) already on the device
            return self._eng.decode_batch(rows[0], rows[1], self.model.kind, form)
        if hasattr(rows, 'values') and hasattr(rows, 'splits'):
            return self._eng.decode_batch(rows, None, self.model.kind, form)
        import numpy as np
        sp = np.zeros(len(rows) + 1, dtype=np.int64)
        np.cumsum([len(r) for r in rows], out=sp[1:])
        flat = np.fromiter((i for r in rows for i in r), dtype=np.int64, count=int(sp[-1]))
        if flat.size and (flat.min() < -2 ** 31 or flat.max() >= 2 ** 31):
            raise IndexError('piece id is out of range.')
        return self._eng.decode_batch(torch.from_numpy(flat.astype(np.int32)), torch.from_numpy(sp), self.model.kind, form)

    def decode_batch(self, id_rows, as_device=False):
        """decode() over a batch: list of id lists, a Ragged from encode_batch(as_device=True), or (ids, splits) device
        tensors -> list[str] (or the TextBatch on the device)"""
        if self.model is None:
            raise ValueError("need model to decode")
        tb = self._ids_to_text(id_rows, C.FORM_DECODE)
        return tb if as_device else tb.to_strings()

    def detokenize_batch(self, id_rows, as_device=False):
        """detokenize(pieces of the ids) over a batch (reference tokenizer.py:236-246)"""
        if self.model is None:
            raise ValueError("need model to detokenize ids")
        tb = self._ids_to_text(id_rows, C.FORM_DETOKENIZE)
        return tb if as_device else tb.to_strings()

    def encode_batch_sharded(self, h_data, h_offsets, group=None, gather=True):
        """encode() of one batch by all the GPUs of the box: every rank of the torch.distributed group (one process per
        GPU) passes the same host arrays (uint8 text, int64 row offsets); each encodes its contiguous share of the rows on
        its own GPU through the pipelined host path and the ragged ids are gathered on the host (shard.encode_sharded)."""
        import numpy as np
        import torch
        from . import shard
        if self.model is None:
            raise ValueError("need model for IDs")

        def enc(d, o):
            hd = torch.from_numpy(np.ascontiguousarray(d)).pin_memory() if d.size else torch.zeros(0, dtype=torch.uint8)
            ho = torch.from_numpy(np.ascontiguousarray(o))
            ids, sp = self.encode_batch_host(hd, ho)
            return ids.numpy().copy(), sp.numpy().copy()
        return shard.encode_sharded(enc, h_data, h_offsets, group, gather)

    def tokenize_batch(self, texts):
        """tokenize() over a batch -> list[list[str]]"""
        if self.model is None:
            return normalize_and_segment_batch(texts, self.normalize_roman, self.clean_hinglish, device=self._device)[1]
        return [self._pieces(ids) for ids in self.encode_batch(texts)]

    def explain_batch(self, texts):
        norm = normalize_batch(texts, self.normalize_roman, self.clean_hinglish, device=self._device)
        ak = segment_akshars_batch(norm, device=self._device)
        cs = detect_code_switches_batch(norm, device=self._device)
        st = analyze_text_composition_batch(norm, device=self._device)
        tk = self.tokenize_batch(texts)
        return [{'original': t, 'normalized': n, 'akshars': a, 'code_switches': c, 'tokens': k, 'stats': s}
                for t, n, a, c, k, s in zip(texts, norm, ak, cs, tk, st)]

    # ------------------------------------------------------------------ helpers
    def _encode_normalized(self, norms):
        if self.model.kind == 0:
            r = self._eng.encode_bpe_batch(norms)
        else:
            r = self._eng.encode_unigram_batch(norms)
        return [x.tolist() for x in r.rows()]

    def _pieces(self, ids):
        return [self.model.token(i) for i in ids]


AksharTokenizer = aksharTokenizer      # the name the reference's tests/test_tokenizer.py:11 imports
