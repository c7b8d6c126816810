"""Batch engine: the host side of the CUDA hot path.

One `Engine` per device wraps a C-ABI context (include/akshar_b200.h).  Inputs are a batch of sentences as
concatenated UTF-8 in HBM (`uint8[total]`) + `int64 row_offsets[n + 1]`; outputs are ragged device tensors
(`Ragged(values, splits)`).  torch is used for device memory and streams only; all arithmetic is in
libakshar_b200.so.  Each method mirrors, for a whole batch, the reference call named in its docstring.
"""
import ctypes
from dataclasses import dataclass

import torch

from . import _lib as C


@dataclass
class Ragged:
    """values[splits[i]:splits[i+1]] belongs to row i; `extra` carries a parallel values tensor (run tags)"""
    values: torch.Tensor
    splits: torch.Tensor
    extra: torch.Tensor = None

    def rows(self):
        v = self.values.cpu().numpy()
        s = self.splits.cpu().numpy()
        return [v[s[i]:s[i + 1]] for i in range(len(s) - 1)]


@dataclass
class TextBatch:
    """concatenated UTF-8 rows resident on the device"""
    data: torch.Tensor         # uint8 [total]
    offsets: torch.Tensor      # int64 [n + 1], absolute byte offsets into data
    begin: int
    end: int

    @property
    def n_rows(self):
        return self.offsets.numel() - 1

    @property
    def n_bytes(self):
        return self.end - self.begin

    def to_strings(self):
        b = self.data.cpu().numpy().tobytes()
        o = self.offsets.cpu().numpy()
        return [b[o[i]:o[i + 1]].decode('utf-8') for i in range(len(o) - 1)]


# why akshar_pair_windows_count refused a pair (the reason in the low 3 bits of result[3])
_PAIR_REFUSED = {1: 'longest_first would cut a sequence to 0 ids: max_length leaves 1 id for both',
                 2: 'stride is not smaller than the length a sequence is cut to',
                 3: 'sequence to truncate too short to respect the provided max_length',
                 4: 'more than 2^31 - 1 windows'}


def _ids_int32(v):
    """int32 ids from int32 ids or compact ids (uint16, or the uint16 bit patterns an int16 tensor holds)"""
    if v.dtype == torch.int16:
        return v.to(torch.int32) & 0xFFFF
    return v.to(torch.int32)


class BatchStatusError(RuntimeError):
    def __init__(self, bits, what):
        self.bits = bits
        names = [n for b, n in ((C.ST_OVERFLOW, 'overflow'), (C.ST_NFC_SEGMENT, 'NFC segment longer than 256 code points'),
                                (C.ST_PATHOLOGICAL, 'look-back limit'), (C.ST_ALPHABET, 'code point outside the closed alphabet'),
                                (C.ST_SPIN, 'tile-prefix spin limit'), (C.ST_WORD, 'word longer than the scratch pool'),
                                (C.ST_INTERNAL, 'internal consistency check (bits 0x%x)' % bits)) if bits & b]
        super().__init__('%s: %s' % (what, ', '.join(names)))


def pack_host(lines, stage=None):
    """list[str] -> (pinned uint8 tensor, pinned int64 offsets) on the host.  `stage` = (data, off) pinned tensors to fill
    instead of pinning fresh memory (Engine.put keeps a pair that only grows: pinning costs more than a small batch)"""
    import numpy as np
    enc = [s.encode('utf-8') for s in lines]
    blob = b''.join(enc)
    total = len(blob)
    if stage is not None and stage[0].numel() >= max(total, 1) and stage[1].numel() >= len(enc) + 1:
        data, off = stage[0][:max(total, 1)], stage[1][:len(enc) + 1]
    else:
        data = torch.empty(max(total, 1), dtype=torch.uint8).pin_memory()
        off = torch.empty(len(enc) + 1, dtype=torch.int64).pin_memory()
    if total:
        data.numpy()[:total] = np.frombuffer(blob, dtype=np.uint8)
    o = off.numpy()
    o[0] = 0
    if enc:
        np.cumsum(np.fromiter((len(e) for e in enc), dtype=np.int64, count=len(enc)), out=o[1:])
    return data[:total], off


class Engine:
    def __init__(self, device=0):
        if not torch.cuda.is_available():
            raise C.AksharCudaError('akshar_b200: no CUDA device; the batch path has no CPU fallback')
        self.lib = C.load()
        self.device = torch.device('cuda', device if isinstance(device, int) else torch.device(device).index or 0)
        h = ctypes.c_void_p()
        rc = self.lib.akshar_ctx_create(self.device.index, ctypes.byref(h))
        self._h = h
        if rc != 0:
            msg = self.lib.akshar_last_error(h).decode() if h else 'out of memory'
            raise C.AksharCudaError('akshar_ctx_create: ' + msg)
        self._ws = None
        self._vocab = {}
        self._pad = {}

    def __del__(self):
        try:
            if getattr(self, '_h', None):
                self.lib.akshar_ctx_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # ------------------------------------------------------------------ plumbing
    def _err(self, rc, what):
        raise C.AksharCudaError('%s: %s (%s)' % (what, self.lib.akshar_status_str(rc).decode(),
                                                 self.lib.akshar_last_error(self._h).decode()))

    def _workspace(self, n_bytes, n_rows, extra=0):
        """`extra` bytes beyond the library's minimum enlarge the temporary output streams (grown after an overflow)"""
        need = self.lib.akshar_workspace_bytes(n_bytes, n_rows) + extra
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need + (need >> 3), dtype=torch.uint8, device=self.device)
        return self._ws

    MAX_TRIES = 5

    def _slot_extra(self, n_bytes):
        """workspace beyond the minimum that gives every 960-byte warp tile the event slots the last call asked for
        (half of a surplus goes to the slots, 20 bytes each; include/akshar_b200.h)"""
        need = getattr(self, '_slots_needed', 0)
        if need <= 256:
            return 0
        cap = 512
        while cap < need:
            cap *= 2                        # slots per warp tile are a power of two
        return 2 * (n_bytes // 960 + 4) * 21 * (cap - 256) + (1 << 20)

    def _stream(self):
        # the stream of THIS engine's device, whatever the caller's current device is
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def launch_count(self):
        return int(self.lib.akshar_launch_count(self._h))

    def timing(self, enable=True):
        """CUDA-event timing of the dominant kernel of each stage (see include/akshar_b200.h)"""
        rc = self.lib.akshar_timing_enable(self._h, 1 if enable else 0)
        if rc != 0:
            self._err(rc, 'akshar_timing_enable')

    def kernel_ms(self, name):
        """duration of kernel `name` in the most recent call, or None if it was not launched"""
        ms = ctypes.c_float()
        rc = self.lib.akshar_timing_read(self._h, C.TIMERS[name], ctypes.byref(ms))
        return float(ms.value) if rc == 0 else None

    def put(self, lines):
        """host list[str] (or (uint8 tensor, int64 offsets) host tensors) -> TextBatch on the device"""
        if isinstance(lines, TextBatch):
            return lines
        staged = False
        if isinstance(lines, (list, tuple)) and (len(lines) == 0 or isinstance(lines[0], str)):
            # the engine's own pinned staging pair (grow-only); the copies out of it are awaited before it is filled again
            stg = self.__dict__.get('_stage')
            ev = self.__dict__.get('_stage_ev')
            if ev is not None:
                ev.synchronize()
            nb = sum(len(s) for s in lines) * 4 + 16                     # UTF-8 is at most 4 bytes per code unit of a str
            if stg is None or stg[0].numel() < nb or stg[1].numel() < len(lines) + 1:
                stg = (torch.empty(max(nb, 1 << 16), dtype=torch.uint8).pin_memory(),
                       torch.empty(max(len(lines) + 1, 1 << 10), dtype=torch.int64).pin_memory())
                self._stage = stg
            data, off = pack_host(lines, stg)
            staged = True
        else:
            data, off = lines
        d = torch.empty(max(data.numel(), 1), dtype=torch.uint8, device=self.device)
        d[:data.numel()].copy_(data, non_blocking=True)
        o = off.to(self.device, non_blocking=True)
        if staged:
            if self.__dict__.get('_stage_ev') is None:
                self._stage_ev = torch.cuda.Event()
            self._stage_ev.record(torch.cuda.current_stream(self.device))
        return TextBatch(d, o, int(off[0]), int(off[-1]))

    def _finish(self, result, what, check):
        if not check:
            return None
        r = result.cpu()
        bits = int(r[2])
        self._slots_needed = int(r[3])        # encoders: event slots per 960 text bytes that were needed (on overflow)
        return int(r[0]), int(r[1]), bits

    # ------------------------------------------------------------------ K1
    def normalize_batch(self, batch, normalize_roman=True, clean_hinglish=True, mode=C.MODE_TILES, capacity=None, check=True):
        """normalize_text over a batch (reference normalize.py:117-148) -> TextBatch"""
        b = self.put(batch)
        flags = (C.NORM_ROMAN if normalize_roman else 0) | (C.NORM_CLEAN if clean_hinglish else 0)
        cap = capacity if capacity is not None else b.n_bytes + (b.n_bytes >> 3) + 1024
        ws = self._workspace(b.n_bytes, b.n_rows)
        for _ in range(self.MAX_TRIES):
            out = torch.empty(max(cap, 1), dtype=torch.uint8, device=self.device)
            out_off = torch.empty(b.n_rows + 1, dtype=torch.int64, device=self.device)
            result = torch.empty(4, dtype=torch.int64, device=self.device)
            rc = self.lib.akshar_normalize_batch(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, b.begin, b.end,
                                                 flags, mode, out.data_ptr(), cap, out_off.data_ptr(), result.data_ptr(),
                                                 ws.data_ptr(), ws.numel(), self._stream())
            if rc != 0:
                self._err(rc, 'akshar_normalize_batch')
            if not check:
                return TextBatch(out, out_off, 0, -1), result
            total, _, bits = self._finish(result, 'normalize', True)
            if bits & C.ST_PATHOLOGICAL and mode == C.MODE_TILES:
                mode = C.MODE_ROWS
                continue
            if bits & C.ST_OVERFLOW:
                cap = total
                continue
            if bits:
                raise BatchStatusError(bits, 'normalize_batch')
            return TextBatch(out, out_off, 0, total)
        raise BatchStatusError(bits, 'normalize_batch (retries exhausted)')

    # ------------------------------------------------------------------ K2 / K3
    def segment_batch(self, batch, clusters=True, matras=False, runs=False, mode=C.MODE_TILES, capacity=None, check=True):
        """segment_akshars / detect_code_switches over a batch (reference segment.py:40-201).
        -> (clusters Ragged | None, runs Ragged | None); values are int32 END byte offsets relative to the row start"""
        b = self.put(batch)
        flags = (C.SEG_CLUSTERS if clusters else 0) | (C.SEG_MATRAS if matras else 0) | (C.SEG_RUNS if runs else 0)
        ccap = rcap = 0
        if clusters:
            ccap = capacity if capacity is not None else (b.n_bytes >> 1) + b.n_rows + 1024
        if runs:
            rcap = capacity if capacity is not None else (b.n_bytes >> 3) + b.n_rows + 1024
        ws = self._workspace(b.n_bytes, b.n_rows)
        for _ in range(self.MAX_TRIES):
            dev = self.device
            ce = torch.empty(max(ccap, 1), dtype=torch.int32, device=dev) if clusters else None
            cs = torch.empty(b.n_rows + 1, dtype=torch.int64, device=dev) if clusters else None
            re_ = torch.empty(max(rcap, 1), dtype=torch.int32, device=dev) if runs else None
            rt = torch.empty(max(rcap, 1), dtype=torch.uint8, device=dev) if runs else None
            rs = torch.empty(b.n_rows + 1, dtype=torch.int64, device=dev) if runs else None
            result = torch.empty(4, dtype=torch.int64, device=dev)
            p = lambda t: t.data_ptr() if t is not None else None
            rc = self.lib.akshar_segment_batch(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, b.begin, b.end, flags,
                                               mode, p(ce), ccap, p(cs), p(re_), p(rt), rcap, p(rs), result.data_ptr(),
                                               ws.data_ptr(), ws.numel(), self._stream())
            if rc != 0:
                self._err(rc, 'akshar_segment_batch')
            if check:
                nc, nr, bits = self._finish(result, 'segment', True)
                if bits & C.ST_PATHOLOGICAL and mode == C.MODE_TILES:
                    mode = C.MODE_ROWS
                    continue
                if bits & C.ST_OVERFLOW:
                    # totals are exact: size the outputs and the temporary streams in the workspace for them
                    ccap, rcap = (max(ccap, nc) if clusters else 0), (max(rcap, nr) if runs else 0)
                    ws = self._workspace(b.n_bytes, b.n_rows, extra=6 * nc + 20 * nr + (1 << 16))
                    continue
                if bits:
                    raise BatchStatusError(bits, 'segment_batch')
                if clusters:
                    ce = ce[:nc]
                if runs:
                    re_, rt = re_[:nr], rt[:nr]
            co = Ragged(ce, cs) if clusters else None
            ro = Ragged(re_, rs, rt) if runs else None
            return (co, ro) if check else (co, ro, result)
        raise BatchStatusError(bits, 'segment_batch (retries exhausted)')

    # ------------------------------------------------------------------ word tokenizers
    def word_tokenize_batch(self, batch, rule=C.WORDS_HINDI, row_flags=False, capacity=None):
        """the word loop of word_tokenize_hindi / word_tokenize_sanskrit (reference segment.py:270-297) over text that is
        already normalized, or `str.split()` (rule WORDS_SPLIT, segment.py:391-393).
        -> (begin, end, splits[, flags]): int32 byte offsets of every token relative to its row start, int64 row splits,
        and with row_flags=True one byte per row: 1 = the row holds a code point of U+0900-097F"""
        b = self.put(batch)
        cap = capacity if capacity is not None else (b.n_bytes >> 2) + b.n_rows + 1024
        ws = self._workspace(b.n_bytes, b.n_rows)
        dev = self.device
        for _ in range(self.MAX_TRIES):
            wb = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
            we = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
            sp = torch.empty(b.n_rows + 1, dtype=torch.int64, device=dev)
            fl = torch.empty(max(b.n_rows, 1), dtype=torch.uint8, device=dev) if row_flags else None
            result = torch.empty(4, dtype=torch.int64, device=dev)
            rc = self.lib.akshar_word_tokenize_batch(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, b.begin, b.end,
                                                     rule, wb.data_ptr(), we.data_ptr(), cap, sp.data_ptr(),
                                                     fl.data_ptr() if row_flags else None, result.data_ptr(), ws.data_ptr(),
                                                     ws.numel(), self._stream())
            if rc != 0:
                self._err(rc, 'akshar_word_tokenize_batch')
            total, _, bits = self._finish(result, 'word_tokenize', True)
            if bits & C.ST_OVERFLOW:
                cap = total
                continue
            if bits:
                raise BatchStatusError(bits, 'word_tokenize_batch')
            out = (wb[:total], we[:total], sp)
            return out + (fl[:b.n_rows],) if row_flags else out
        raise BatchStatusError(bits, 'word_tokenize_batch (retries exhausted)')

    # ------------------------------------------------------------------ file bytes -> rows
    def lines_batch(self, d_file, n_bytes, row_capacity=None):
        """the lines of a text file as rows (reference cli.py:165-190: readlines / strip / skip empty) from the file's bytes
        on the device -> TextBatch"""
        dev = self.device
        rcap = row_capacity if row_capacity is not None else n_bytes // 24 + 1024
        for _ in range(self.MAX_TRIES):
            need = self.lib.akshar_lines_workspace_bytes(n_bytes, rcap)
            if self._ws is None or self._ws.numel() < need:
                self._ws = None
                self._ws = torch.empty(need + (need >> 3), dtype=torch.uint8, device=dev)
            ws = self._ws
            out = torch.empty(max(n_bytes, 1), dtype=torch.uint8, device=dev)
            off = torch.empty(rcap + 1, dtype=torch.int64, device=dev)
            result = torch.empty(4, dtype=torch.int64, device=dev)
            rc = self.lib.akshar_lines_batch(self._h, d_file.data_ptr(), n_bytes, out.data_ptr(), n_bytes, off.data_ptr(), rcap,
                                             result.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
            if rc != 0:
                self._err(rc, 'akshar_lines_batch')
            r = result.cpu()
            rows, total, bits = int(r[0]), int(r[1]), int(r[2])
            if bits & C.ST_OVERFLOW:
                rcap = rows
                continue
            if bits:
                raise BatchStatusError(bits, 'lines_batch')
            return TextBatch(out, off[:rows + 1], 0, total)
        raise BatchStatusError(bits, 'lines_batch (retries exhausted)')

    def join_rows(self, batch, sep=0x0A):
        """every row followed by `sep`, as one uint8 tensor on the device (the file preprocess_corpus writes)"""
        b = self.put(batch)
        out = torch.empty(max(b.n_bytes + b.n_rows, 1), dtype=torch.uint8, device=self.device)
        rc = self.lib.akshar_join_rows(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, sep, out.data_ptr(), self._stream())
        if rc != 0:
            self._err(rc, 'akshar_join_rows')
        return out[:b.n_bytes + b.n_rows]

    # ------------------------------------------------------------------ per-sentence statistics, cluster merging
    def composition_batch(self, batch):
        """-> int32 [n_rows, 5] on the device: akshars, script runs, code points, code points in devanagari / roman runs"""
        b = self.put(batch)
        clusters, runs = self.segment_batch(b, clusters=True, runs=True)
        stats = torch.empty((max(b.n_rows, 1), 5), dtype=torch.int32, device=self.device)
        rc = self.lib.akshar_composition_batch(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, clusters.splits.data_ptr(),
                                               runs.values.data_ptr(), runs.extra.data_ptr(), runs.splits.data_ptr(),
                                               stats.data_ptr(), self._stream())
        if rc != 0:
            self._err(rc, 'akshar_composition_batch')
        return stats[:b.n_rows]

    def merge_clusters_batch(self, batch, clusters, rule):
        """the cluster-merging feature wrappers (reference features.py:28-55, 173-206) -> Ragged like `clusters`"""
        b = self.put(batch)
        n = clusters.values.numel()
        need = self.lib.akshar_merge_workspace_bytes(n)
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need + (need >> 3), dtype=torch.uint8, device=self.device)
        ws = self._ws
        out = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)
        sp = torch.empty(b.n_rows + 1, dtype=torch.int64, device=self.device)
        result = torch.empty(4, dtype=torch.int64, device=self.device)
        rc = self.lib.akshar_merge_clusters_batch(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, clusters.values.data_ptr(),
                                                  clusters.splits.data_ptr(), n, rule, out.data_ptr(), n, sp.data_ptr(),
                                                  result.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
        if rc != 0:
            self._err(rc, 'akshar_merge_clusters_batch')
        total, _, bits = self._finish(result, 'merge_clusters', True)
        if bits:
            raise BatchStatusError(bits, 'merge_clusters_batch')
        return Ragged(out[:total], sp)

    # ------------------------------------------------------------------ ids -> text
    def decode_batch(self, ids, splits, kind, form=C.FORM_DECODE, capacity=None):
        """aksharTokenizer.decode / detokenize over a batch of id rows (reference tokenizer.py:195-246) -> TextBatch.
        ids: device int32 (or uint16) tensor, or a Ragged from encode; splits: int64 [n_rows + 1] positions in ids"""
        if isinstance(ids, Ragged):
            ids, splits = ids.values, ids.splits
        dev = self.device
        ids = ids.to(dev)
        splits = splits.to(dev)
        if ids.dtype not in (torch.int32, torch.uint16, torch.int16):
            ids = ids.to(torch.int32)
        n_ids, n_rows = ids.numel(), splits.numel() - 1
        need = self.lib.akshar_decode_workspace_bytes(n_ids, n_rows)
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need + (need >> 3), dtype=torch.uint8, device=dev)
        ws = self._ws
        cap = capacity if capacity is not None else 6 * n_ids + 1024
        for _ in range(self.MAX_TRIES):
            out = torch.empty(max(cap, 1), dtype=torch.uint8, device=dev)
            out_off = torch.empty(n_rows + 1, dtype=torch.int64, device=dev)
            result = torch.empty(4, dtype=torch.int64, device=dev)
            rc = self.lib.akshar_decode_batch(self._h, kind, form, ids.data_ptr(), 0 if ids.dtype == torch.int32 else 1, n_ids,
                                              splits.data_ptr(), n_rows, out.data_ptr(), cap, out_off.data_ptr(), result.data_ptr(),
                                              ws.data_ptr(), ws.numel(), self._stream())
            if rc != 0:
                self._err(rc, 'akshar_decode_batch')
            total, _, bits = self._finish(result, 'decode', True)
            if bits & C.ST_BAD_ID:
                raise IndexError('piece id is out of range.')         # what SentencePiece's DecodeIds raises
            if bits & C.ST_OVERFLOW:
                cap = total
                continue
            if bits:
                raise BatchStatusError(bits, 'decode_batch')
            return TextBatch(out, out_off, 0, total)
        raise BatchStatusError(bits, 'decode_batch (retries exhausted)')

    # ------------------------------------------------------------------ ids -> model-ready windows
    def pad_id(self, kind):
        """id of the model's pad piece: the '<pad>' token of a BPE model, the '<pad>' control piece of a SentencePiece model
        (which has none unless it was trained with pad_id >= 0); None without one"""
        if kind not in self._pad:
            want = 1 if kind == 0 else 3                          # BPE special token / SentencePiece CONTROL piece
            self._pad[kind] = next((i for i, (p, t) in enumerate(self.vocab(kind)[1]) if p == '<pad>' and t == want), None)
        return self._pad[kind]

    def windows_batch(self, ids, kind, max_length=None, padding='longest', truncation=False, stride=0,
                      return_overflowing_tokens=False, pad_to_multiple_of=None, padding_side='right', truncation_side='right',
                      pad_id=None, pair_ids=None):
        """encoder output -> the dense batch a model takes, bit-exact with HF tokenizers' truncation (with stride and
        overflowing windows) and padding, and with what transformers' `tokenizer(texts, truncation=..., max_length=...,
        stride=..., return_overflowing_tokens=..., padding=..., pad_to_multiple_of=..., return_tensors='pt')` returns
        for the model's `<s> $A </s>` template (the rule: include/akshar_b200.h, akshar_windows_count).
        ids: a Ragged of model `kind` from the encoders (int32 or uint16 values), or a (values, splits) pair.
        padding: 'longest' (the longest window of the call) or 'max_length'; the width is then rounded up to
        pad_to_multiple_of.  pad_id defaults to the model's pad piece.
        -> dict of int64 device tensors: input_ids [N, L], attention_mask [N, L], and with return_overflowing_tokens
        overflow_to_sample_mapping [N] (the row of every window; windows are in row order, window 0 first).
        pair_ids: the second sequences of sentence pairs (row i of ids with row i of pair_ids), as ids; the windows are
        then those of `tokenizer(texts, text_pair, ...)` through the model's pair template (akshar_pair_windows_count),
        and truncation takes True / 'longest_first', 'only_first', 'only_second', or False / 'do_not_truncate'.
        Raises ValueError where HF would misbehave (see the header) and for ids the encoder of this model did not produce.
        One read-back of the result block (N, longest window, status); nothing else synchronises."""
        values, splits = (ids.values, ids.splits) if isinstance(ids, Ragged) else ids
        only = 0
        if pair_ids is not None:
            strategies = {'longest_first': 0, 'only_first': C.WIN_ONLY_FIRST, 'only_second': C.WIN_ONLY_SECOND}
            if isinstance(truncation, str):
                if truncation != 'do_not_truncate' and truncation not in strategies:
                    raise ValueError("truncation must be True, False, 'longest_first', 'only_first', 'only_second' or "
                                     "'do_not_truncate'")
                only = strategies.get(truncation, 0)
                truncation = truncation != 'do_not_truncate'
        if padding not in ('longest', 'max_length'):
            raise ValueError("padding must be 'longest' or 'max_length'")
        if padding_side not in ('left', 'right') or truncation_side not in ('left', 'right'):
            raise ValueError("padding_side and truncation_side must be 'left' or 'right'")
        if (truncation or padding == 'max_length') and max_length is None:
            raise ValueError('truncation and padding to max_length need max_length')
        if not truncation and (stride or return_overflowing_tokens):
            raise ValueError('stride and return_overflowing_tokens need truncation')
        if pad_to_multiple_of is not None and pad_to_multiple_of < 1:
            raise ValueError('pad_to_multiple_of must be positive')
        if pad_id is None:
            pad_id = self.pad_id(kind)
            if pad_id is None:
                raise ValueError('the model has no pad piece: pass pad_id')
        dev = self.device
        values, splits = values.to(dev), splits.to(dev, torch.int64)
        if values.dtype not in (torch.int32, torch.uint16, torch.int16):
            values = values.to(torch.int32)
        if pair_ids is not None:
            values_b, splits_b = (pair_ids.values, pair_ids.splits) if isinstance(pair_ids, Ragged) else pair_ids
            values_b, splits_b = values_b.to(dev), splits_b.to(dev, torch.int64)
            if values_b.dtype not in (torch.int32, torch.uint16, torch.int16):
                values_b = values_b.to(torch.int32)
            if (values.dtype == torch.int32) != (values_b.dtype == torch.int32):
                values, values_b = _ids_int32(values), _ids_int32(values_b)
            if splits_b.numel() != splits.numel():
                raise ValueError('ids and pair_ids must hold the same number of rows')
            if values_b.numel() >= 2 ** 31:
                raise ValueError('windows_batch takes fewer than 2^31 ids per call')
        if values.numel() >= 2 ** 31:
            raise ValueError('windows_batch takes fewer than 2^31 ids per call')
        u16 = 0 if values.dtype == torch.int32 else 1
        n_rows = splits.numel() - 1
        flags = ((C.WIN_TRUNCATE if truncation else 0) | (C.WIN_OVERFLOW if return_overflowing_tokens else 0) |
                 (C.WIN_TRUNC_LEFT if truncation_side == 'left' else 0) | (C.WIN_PAD_LEFT if padding_side == 'left' else 0) | only)
        ml = max_length if max_length is not None else 0
        need = self.lib.akshar_windows_workspace_bytes(n_rows)
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need + (need >> 3), dtype=torch.uint8, device=dev)
        wsplits = torch.empty(n_rows + 1, dtype=torch.int64, device=dev)
        result = torch.empty(4, dtype=torch.int64, device=dev)
        if pair_ids is None:
            rc = self.lib.akshar_windows_count(self._h, kind, values.data_ptr(), u16, splits.data_ptr(), n_rows, ml, stride, flags,
                                               wsplits.data_ptr(), result.data_ptr(), self._ws.data_ptr(), self._ws.numel(),
                                               self._stream())
        else:
            rc = self.lib.akshar_pair_windows_count(self._h, kind, values.data_ptr(), splits.data_ptr(), values_b.data_ptr(),
                                                    splits_b.data_ptr(), u16, n_rows, ml, stride, flags, wsplits.data_ptr(),
                                                    result.data_ptr(), self._ws.data_ptr(), self._ws.numel(), self._stream())
        if rc == C.E_ARG:
            raise ValueError(self.lib.akshar_last_error(self._h).decode())
        if rc != 0:
            self._err(rc, 'akshar_pair_windows_count' if pair_ids is not None else 'akshar_windows_count')
        n, longest, bits, refused = (int(x) for x in result.cpu())
        if bits & C.ST_TEMPLATE:
            raise ValueError('a row does not begin / end with the template ids of the model: not ids of its encoder')
        if bits & C.ST_PAIR_TRUNC:
            if refused & 7 == 5:
                raise ValueError('the %d pairs give more than 2^31 - 1 windows in all: window fewer pairs per call' % n_rows)
            raise ValueError('pair %d: %s' % (refused >> 3, _PAIR_REFUSED.get(refused & 7, 'cannot be truncated as asked')))
        if bits:
            raise BatchStatusError(bits, 'windows_batch')
        width = max_length if padding == 'max_length' else longest
        if pad_to_multiple_of:
            width = -(-width // pad_to_multiple_of) * pad_to_multiple_of
        if longest > width:
            raise ValueError('a row of %d ids is longer than max_length = %d: truncate it' % (longest, max_length))
        out_ids = torch.empty((n, width), dtype=torch.int64, device=dev)
        mask = torch.empty((n, width), dtype=torch.int64, device=dev)
        sample = torch.empty(n, dtype=torch.int64, device=dev)
        if pair_ids is None:
            rc = self.lib.akshar_windows_write(self._h, kind, values.data_ptr(), u16, splits.data_ptr(), wsplits.data_ptr(), n_rows,
                                               n, ml, stride, flags, width, pad_id, out_ids.data_ptr(), mask.data_ptr(),
                                               sample.data_ptr(), self._stream())
        else:
            rc = self.lib.akshar_pair_windows_write(self._h, kind, values.data_ptr(), splits.data_ptr(), values_b.data_ptr(),
                                                    splits_b.data_ptr(), u16, wsplits.data_ptr(), n_rows, n, ml, stride, flags, width,
                                                    pad_id, out_ids.data_ptr(), mask.data_ptr(), sample.data_ptr(), self._stream())
        if rc != 0:
            self._err(rc, 'akshar_pair_windows_write' if pair_ids is not None else 'akshar_windows_write')
        out = {'input_ids': out_ids, 'attention_mask': mask}
        if return_overflowing_tokens:
            out['overflow_to_sample_mapping'] = sample
        return out

    # ------------------------------------------------------------------ ids -> packed language-model batches
    def pack_batch(self, ids, block_size, eos_id=None, carry=None, separator_id=-100, return_position_ids=True,
                   return_seq_idx=False, return_flash_attn_kwargs=False):
        """encoder output -> fixed blocks of `block_size` ids for causal-LM training without padding: the rows (one per
        document, each followed by `eos_id` when one is given) concatenated after `carry` and cut into blocks as
        transformers' run_clm.py `group_texts` cuts them, with the keys transformers'
        DataCollatorWithFlattening(return_position_ids, separator_id, return_flash_attn_kwargs, return_seq_idx) returns
        for the pieces the blocks and document starts cut the stream into (the rule: include/akshar_b200.h,
        akshar_pack_count).  ids: a Ragged from the encoders (int32 or uint16 values), or a (values, splits) pair.
        -> (batch, rest).  batch: input_ids, labels, position_ids (with return_position_ids) int64 [N, L] and seq_idx int32
        [N, L] (with return_seq_idx); `.view(1, -1)` is the collator's layout, and with return_flash_attn_kwargs
        cu_seq_lens_q / cu_seq_lens_k (int32 [pieces + 1], positions in that flattened layout) and max_length_q /
        max_length_k (Python ints).  rest: the ids after the last whole block (fewer than block_size) as a device Ragged
        (int32 values, int64 splits at document starts); pass it as the next call's `carry` and packing in chunks gives
        the blocks of packing in one call.  Raises ValueError for block_size < 1, eos_id outside [0, 2^31), a carry not
        of the returned form and a stream of 2^31 ids or more.  One read-back of the result block; nothing else
        synchronises."""
        if isinstance(block_size, bool) or not isinstance(block_size, int) or block_size < 1:
            raise ValueError('block_size must be an int of at least 1')
        if eos_id is not None and (isinstance(eos_id, bool) or not isinstance(eos_id, int) or not 0 <= eos_id < 2 ** 31):
            raise ValueError('eos_id must be None or an int in [0, 2^31)')
        if isinstance(separator_id, bool) or not isinstance(separator_id, int) or not -2 ** 63 <= separator_id < 2 ** 63:
            raise ValueError('separator_id must be an int64')
        dev = self.device
        values, splits = (ids.values, ids.splits) if isinstance(ids, Ragged) else ids
        values, splits = values.to(dev), splits.to(dev, torch.int64)
        if values.dtype not in (torch.int32, torch.uint16, torch.int16):
            values = values.to(torch.int32)
        if splits.dim() != 1 or splits.numel() < 1:
            raise ValueError('splits must be an int64 vector of n_rows + 1 positions')
        if carry is None:
            cv = cs = None
            n_carry = 0
        else:
            if isinstance(carry, Ragged):
                cv, cs = carry.values, carry.splits
            elif isinstance(carry, (tuple, list)) and len(carry) == 2:
                cv, cs = carry
            else:
                cv = cs = None
            if not (isinstance(cv, torch.Tensor) and isinstance(cs, torch.Tensor) and cv.dtype == torch.int32 and
                    cs.dtype == torch.int64 and cv.dim() == 1 and cs.dim() == 1 and cs.numel() >= 1 and cv.device == dev and
                    cs.device == dev):
                raise ValueError('carry must be the rest returned by pack_batch: (int32 values, int64 splits) on %s' % dev)
            n_carry = cs.numel() - 1
        if values.numel() + (cv.numel() if cv is not None else 0) >= 2 ** 31:
            raise ValueError('pack_batch takes a stream of fewer than 2^31 ids per call (cu_seq_lens and seq_idx are int32)')
        u16 = 0 if values.dtype == torch.int32 else 1
        n_rows = splits.numel() - 1
        eos = -1 if eos_id is None else eos_id
        need = self.lib.akshar_pack_workspace_bytes(n_rows + n_carry)
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need + (need >> 3), dtype=torch.uint8, device=dev)
        ws = self._ws
        p = lambda t: t.data_ptr() if t is not None and t.numel() else None
        args = (values.data_ptr() if values.numel() else None, u16, splits.data_ptr(), n_rows, p(cv), p(cs) if n_carry else None,
                n_carry, block_size, eos)
        result = torch.empty(8, dtype=torch.int64, device=dev)
        rc = self.lib.akshar_pack_count(self._h, *args, result.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
        if rc == C.E_ARG:
            raise ValueError(self.lib.akshar_last_error(self._h).decode())
        if rc != 0:
            self._err(rc, 'akshar_pack_count')
        n, n_pieces, bits, longest, total, n_frags, _, _ = (int(x) for x in result.cpu())
        if bits & C.ST_PACK_LONG:
            raise ValueError('the stream of this call holds %d ids: pack_batch takes fewer than 2^31 per call (cu_seq_lens '
                             'and seq_idx are int32)' % total)
        if bits:
            raise BatchStatusError(bits, 'pack_batch')
        L = block_size
        out_ids = torch.empty((n, L), dtype=torch.int64, device=dev)
        labels = torch.empty((n, L), dtype=torch.int64, device=dev)
        pos = torch.empty((n, L), dtype=torch.int64, device=dev) if return_position_ids else None
        seq = torch.empty((n, L), dtype=torch.int32, device=dev) if return_seq_idx else None
        cu = torch.empty(n_pieces + 1, dtype=torch.int32, device=dev) if return_flash_attn_kwargs else None
        rest_ids = torch.empty(total - n * L, dtype=torch.int32, device=dev)
        rest_splits = torch.empty(n_frags + 1, dtype=torch.int64, device=dev)
        q = lambda t: t.data_ptr() if t is not None else None
        rc = self.lib.akshar_pack_write(self._h, *args, separator_id, total, n_pieces, n_frags, q(out_ids) if n else None,
                                        q(labels) if n else None, q(pos) if n else None, q(seq) if n else None, q(cu),
                                        p(rest_ids), rest_splits.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
        if rc != 0:
            self._err(rc, 'akshar_pack_write')
        batch = {'input_ids': out_ids, 'labels': labels}
        if return_position_ids:
            batch['position_ids'] = pos
        if return_seq_idx:
            batch['seq_idx'] = seq
        if return_flash_attn_kwargs:
            batch['cu_seq_lens_q'] = batch['cu_seq_lens_k'] = cu
            batch['max_length_q'] = batch['max_length_k'] = longest
        return batch, Ragged(rest_ids, rest_splits)

    def segment_masks(self, batch, clusters=True, matras=False, runs=False, out=None, check=True):
        """segment_batch with AKSHAR_SEG_MASK: the boundaries as bit masks, one bit per text byte (bit p - begin set when a
        cluster / run ends at byte p) -> dict(cluster=uint32 [W] | None, run=uint32 [W] | None, tags=uint32 [2, W] | None,
        n_clusters, n_runs); W = (bytes + 32) // 32.  `out` may hold preallocated tensors under the same keys."""
        b = self.put(batch)
        flags = (C.SEG_CLUSTERS if clusters else 0) | (C.SEG_MATRAS if matras else 0) | (C.SEG_RUNS if runs else 0) | C.SEG_MASK
        W = (b.n_bytes + 32) // 32
        dev = self.device
        out = out or {}
        cm = (out.get('cluster') if out.get('cluster') is not None else torch.empty(W, dtype=torch.int32, device=dev)) if clusters else None
        rm = (out.get('run') if out.get('run') is not None else torch.empty(W, dtype=torch.int32, device=dev)) if runs else None
        tg = (out.get('tags') if out.get('tags') is not None else torch.empty((2, W), dtype=torch.int32, device=dev)) if runs else None
        ws = self._workspace(b.n_bytes, b.n_rows)
        result = torch.empty(4, dtype=torch.int64, device=dev)
        p = lambda t: t.data_ptr() if t is not None else None
        rc = self.lib.akshar_segment_batch(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, b.begin, b.end, flags,
                                           C.MODE_TILES, p(cm), W, None, p(rm), p(tg), W, None, result.data_ptr(),
                                           ws.data_ptr(), ws.numel(), self._stream())
        if rc != 0:
            self._err(rc, 'akshar_segment_batch')
        if check:
            bits = int(result.cpu()[2])
            if bits & C.ST_PATHOLOGICAL:
                # a bounded look-back gave up (thousands of Extend characters in a row): the offset form knows the
                # row-sequential mode; its ends are turned into the same masks
                cl, ru = self.segment_batch(b, clusters=clusters, matras=matras, runs=runs)
                return self._masks_from_ragged(b, cl, ru, W)
            if bits:
                raise BatchStatusError(bits, 'segment_masks')
        return {'cluster': cm, 'run': rm, 'tags': tg, 'result': result, 'words': W}

    def _masks_from_ragged(self, b, cl, ru, W):
        dev = self.device
        off = b.offsets - b.begin

        def words(rag, keep=None):
            rows = torch.repeat_interleave(torch.arange(b.n_rows, device=dev), rag.splits[1:] - rag.splits[:-1])
            pos = off[rows] + rag.values.to(torch.int64)
            if keep is not None:
                pos = pos[keep]
            bits = torch.zeros(W * 32, dtype=torch.int64, device=dev)
            bits[pos] = 1
            w = (bits.view(W, 32) << torch.arange(32, device=dev, dtype=torch.int64)).sum(dim=1)
            return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32)

        out = {'cluster': None, 'run': None, 'tags': None, 'words': W}
        res = torch.zeros(4, dtype=torch.int64, device=dev)
        if cl is not None:
            out['cluster'] = words(cl)
            res[0] = cl.values.numel()
        if ru is not None:
            out['run'] = words(ru)
            t = ru.extra
            out['tags'] = torch.stack([words(ru, (t == 1) | (t == 255)), words(ru, (t == 4) | (t == 255))])
            res[1] = ru.values.numel()
        out['result'] = res
        return out

    def normalize_segment_batch(self, batch, normalize_roman=True, clean_hinglish=True, clusters=True, matras=False, runs=True,
                                check=True):
        """normalize_text -> akshars / script runs in ONE library call (nothing read back in between): -> (normalized
        TextBatch, masks dict as segment_masks returns it).  check=False: no read-back at all (the caller looks at
        masks['result'] itself: [clusters, runs, status bits, normalized bytes])"""
        b = self.put(batch)
        nflags = (C.NORM_ROMAN if normalize_roman else 0) | (C.NORM_CLEAN if clean_hinglish else 0)
        sflags = (C.SEG_CLUSTERS if clusters else 0) | (C.SEG_MATRAS if matras else 0) | (C.SEG_RUNS if runs else 0)
        dev = self.device
        cap = b.n_bytes + (b.n_bytes >> 3) + 1024
        for _ in range(self.MAX_TRIES):
            W = (cap + 32) // 32
            ws = self._workspace(max(cap, b.n_bytes), b.n_rows)
            out = torch.empty(max(cap, 1), dtype=torch.uint8, device=dev)
            out_off = torch.empty(b.n_rows + 1, dtype=torch.int64, device=dev)
            cm = torch.empty(W, dtype=torch.int32, device=dev) if clusters else None
            rm = torch.empty(W, dtype=torch.int32, device=dev) if runs else None
            tg = torch.empty((2, W), dtype=torch.int32, device=dev) if runs else None
            result = torch.empty(4, dtype=torch.int64, device=dev)
            p = lambda t: t.data_ptr() if t is not None else None
            rc = self.lib.akshar_normalize_segment_batch(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, b.begin, b.end,
                                                         nflags, sflags, out.data_ptr(), cap, out_off.data_ptr(), p(cm), p(rm), p(tg), W,
                                                         result.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
            if rc != 0:
                self._err(rc, 'akshar_normalize_segment_batch')
            if not check:
                return TextBatch(out, out_off, 0, -1), {'cluster': cm, 'run': rm, 'tags': tg, 'result': result, 'words': W}
            r = result.cpu()
            bits, total = int(r[2]), int(r[3])
            if bits & C.ST_PATHOLOGICAL:
                # a bounded look-back gave up: the two stages one after the other, the first in its row-sequential mode
                norm = self.normalize_batch(b, normalize_roman, clean_hinglish)
                return norm, self.segment_masks(norm, clusters, matras, runs)
            if bits & C.ST_OVERFLOW:
                cap = total + 1024
                continue
            if bits:
                raise BatchStatusError(bits, 'normalize_segment_batch')
            return TextBatch(out, out_off, 0, total), {'cluster': cm, 'run': rm, 'tags': tg, 'result': result, 'words': W}
        raise BatchStatusError(bits, 'normalize_segment_batch (retries exhausted)')

    def pipeline_host_pipelined(self, h_data, h_off, normalize_roman=True, clean_hinglish=True, matras=False, chunk_bytes=None):
        """normalize_text -> akshars -> script runs of a batch held in pinned host memory, results in pinned host memory
        (`PipelineOut`): the rows go through the device in chunks, the copy in of chunk k + 1, the kernels of chunk k and the
        copy out of chunk k - 2 overlap on three streams.  What crosses the link back is the normalized text, its row
        offsets and 4 bits per normalized byte of boundary masks.  The results live in buffers the engine reuses (valid
        until the next call)."""
        import os
        import numpy as np
        from . import shard
        if chunk_bytes is None:
            chunk_bytes = int(os.environ.get('AKSHAR_CHUNK_MB', '64')) << 20
        dev = self.device
        n_rows = h_off.numel() - 1
        off_np = h_off.numpy()
        total_bytes = int(off_np[-1] - off_np[0])
        ranges = shard.chunk_rows(off_np, chunk_bytes)
        max_b = max(int(off_np[hi] - off_np[lo]) for lo, hi in ranges)
        max_r = max(hi - lo for lo, hi in ranges)
        nflags = (C.NORM_ROMAN if normalize_roman else 0) | (C.NORM_CLEAN if clean_hinglish else 0)
        sflags = C.SEG_CLUSTERS | C.SEG_RUNS | (C.SEG_MATRAS if matras else 0)
        ncap = max_b + (max_b >> 3) + 1024
        W = (ncap + 32) // 32
        ws = self._workspace(ncap, max_r)
        pc = self.__dict__.setdefault('_pipe2_cache', {})
        est_b = total_bytes + (total_bytes >> 4) + 4096
        est_w = (est_b + 32) // 32 + len(ranges) + 8
        # pinned result buffers are kept and only ever grow
        if pc.get('norm') is None or pc['norm'].numel() < est_b:
            pc['norm'] = torch.empty(est_b + (est_b >> 4), dtype=torch.uint8).pin_memory()
        if pc.get('off') is None or pc['off'].numel() < n_rows + 1:
            pc['off'] = torch.empty(n_rows + 1 + (n_rows >> 4), dtype=torch.int64).pin_memory()
        if pc.get('masks') is None or pc['masks'].shape[1] < est_w:
            pc['masks'] = torch.empty((4, est_w + (est_w >> 4)), dtype=torch.int32).pin_memory()
        h_norm, h_noff, h_masks = pc['norm'], pc['off'][:n_rows + 1], pc['masks']
        if 'streams' not in pc:
            pc['streams'] = tuple(torch.cuda.Stream(device=dev) for _ in range(3))
        s_in, s_comp, s_out = pc['streams']
        NSETS = 3
        key = (max_b, max_r)
        sets = pc.get('sets') if pc.get('sets_key') == key else None
        if sets is None:
            sets = [{
                'text': torch.empty(max(max_b, 1), dtype=torch.uint8, device=dev),
                'off': torch.empty(max_r + 1, dtype=torch.int64, device=dev),
                'norm': torch.empty(max(ncap, 1), dtype=torch.uint8, device=dev),
                'norm_off': torch.empty(max_r + 1, dtype=torch.int64, device=dev),
                'masks': torch.empty((4, W), dtype=torch.int32, device=dev),
                'result': torch.empty(4, dtype=torch.int64, device=dev),
                'ev_in': torch.cuda.Event(), 'ev_comp': torch.cuda.Event(), 'ev_out': torch.cuda.Event(),
            } for _ in range(NSETS)]
        pc['sets'], pc['sets_key'] = sets, key
        cur = torch.cuda.current_stream(dev)
        for st in (s_in, s_comp, s_out):
            st.wait_stream(cur)
        chunk_rows = np.array([lo for lo, _ in ranges] + [n_rows], dtype=np.int64)
        chunk_b = np.zeros(len(ranges) + 1, dtype=np.int64)
        chunk_w = np.zeros(len(ranges) + 1, dtype=np.int64)
        state = {'b': 0, 'w': 0, 'c': 0, 'r': 0}

        def finish(k):
            lo, hi = ranges[k]
            S = sets[k % NSETS]
            with torch.cuda.stream(s_out):
                s_out.wait_event(S['ev_comp'])
                r = S['result'].cpu()
                bits, nb = int(r[2]), int(r[3])
                norm, noff, masks = S['norm'], S['norm_off'], S['masks']
                nc, nr = int(r[0]), int(r[1])
                if bits:
                    # this chunk again through the plain path (larger capacities / the row-sequential normalizer)
                    self.redone_chunks = getattr(self, 'redone_chunks', 0) + 1
                    b0, b1 = int(off_np[lo]), int(off_np[hi])
                    nbatch, mk = self.normalize_segment_batch((h_data[b0:b1], h_off[lo:hi + 1] - b0), normalize_roman, clean_hinglish,
                                                              True, matras, True)
                    rr = mk['result'].cpu()
                    nc, nr, nb = int(rr[0]), int(rr[1]), nbatch.end
                    norm, noff = nbatch.data, nbatch.offsets
                    masks = torch.stack([mk['cluster'], mk['run'], mk['tags'][0], mk['tags'][1]])
                nw = (nb + 32) // 32
                if state['b'] + nb > h_norm.numel() or state['w'] + nw > h_masks.shape[1]:
                    raise BatchStatusError(C.ST_OVERFLOW, 'pipeline_host_pipelined: the normalized text grew beyond the pinned result buffers')
                h_norm[state['b']:state['b'] + nb].copy_(norm[:nb], non_blocking=True)
                h_noff[lo + 1:hi + 1].copy_(noff[1:hi - lo + 1] + state['b'], non_blocking=True)
                for pl in range(4):              # plane by plane: contiguous copies (a strided 2-D copy would be staged)
                    h_masks[pl, state['w']:state['w'] + nw].copy_(masks[pl, :nw], non_blocking=True)
                S['ev_out'].record(s_out)
                chunk_b[k], chunk_w[k] = state['b'], state['w']
                state['b'] += nb
                state['w'] += nw
                state['c'] += nc
                state['r'] += nr

        h_noff[0] = 0
        try:
            for k, (lo, hi) in enumerate(ranges):
                S = sets[k % NSETS]
                b0, b1 = int(off_np[lo]), int(off_np[hi])
                nb, nr = b1 - b0, hi - lo
                with torch.cuda.stream(s_in):
                    if k >= NSETS:
                        s_in.wait_event(S['ev_comp'])
                    S['text'][:nb].copy_(h_data[b0:b1], non_blocking=True)
                    S['off'][:nr + 1].copy_(h_off[lo:hi + 1], non_blocking=True)
                    S['ev_in'].record(s_in)
                with torch.cuda.stream(s_comp):
                    s_comp.wait_event(S['ev_in'])
                    if k >= NSETS:
                        s_comp.wait_event(S['ev_out'])
                    m = S['masks']
                    rc = self.lib.akshar_normalize_segment_batch(
                        self._h, S['text'].data_ptr() - b0, S['off'].data_ptr(), nr, b0, b1, nflags, sflags, S['norm'].data_ptr(), ncap,
                        S['norm_off'].data_ptr(), m[0].data_ptr(), m[1].data_ptr(), m[2].data_ptr(), W, S['result'].data_ptr(),
                        ws.data_ptr(), ws.numel(), ctypes.c_void_p(s_comp.cuda_stream))
                    if rc != 0:
                        self._err(rc, 'akshar_normalize_segment_batch')
                    S['ev_comp'].record(s_comp)
                if k >= 2:
                    finish(k - 2)
            for k in range(max(0, len(ranges) - 2), len(ranges)):
                finish(k)
        finally:
            for st in (s_in, s_comp, s_out):
                cur.wait_stream(st)
            torch.cuda.synchronize(dev)
        chunk_b[len(ranges)], chunk_w[len(ranges)] = state['b'], state['w']
        return PipelineOut(h_norm[:state['b']], h_noff, h_masks[0], h_masks[1], h_masks[2], h_masks[3], chunk_rows, chunk_b, chunk_w,
                           state['c'], state['r'])

    # ------------------------------------------------------------------ K1b
    def signature_batch(self, batch):
        """roman_phonetic_signature over a batch of words, one per row (reference normalize.py:59-89) -> TextBatch"""
        b = self.put(batch)
        cap = b.n_bytes + (b.n_bytes >> 1) + 16
        ws = self._workspace(b.n_bytes, b.n_rows)
        out = torch.empty(max(cap, 1), dtype=torch.uint8, device=self.device)
        out_off = torch.empty(b.n_rows + 1, dtype=torch.int64, device=self.device)
        result = torch.empty(4, dtype=torch.int64, device=self.device)
        rc = self.lib.akshar_signature_batch(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, b.begin, b.end,
                                             out.data_ptr(), cap, out_off.data_ptr(), result.data_ptr(), ws.data_ptr(),
                                             ws.numel(), self._stream())
        if rc != 0:
            self._err(rc, 'akshar_signature_batch')
        total, _, bits = self._finish(result, 'signature', True)
        if bits:
            raise BatchStatusError(bits, 'signature_batch')
        return TextBatch(out, out_off, 0, total)

    # ------------------------------------------------------------------ K4
    def load_bpe(self, path_or_bytes):
        """Tokenizer.from_file for the CUDA path (reference tokenizer.py:96-98)"""
        data = path_or_bytes if isinstance(path_or_bytes, (bytes, bytearray)) else open(path_or_bytes, 'rb').read()
        rc = self.lib.akshar_load_bpe_json(self._h, bytes(data), len(data))
        if rc != 0:
            self._err(rc, 'akshar_load_bpe_json')
        self._vocab.pop(0, None)
        self._pad.pop(0, None)

    def load_spm(self, path_or_bytes):
        """SentencePieceProcessor.Load for the CUDA path (reference tokenizer.py:88-91)"""
        data = path_or_bytes if isinstance(path_or_bytes, (bytes, bytearray)) else open(path_or_bytes, 'rb').read()
        rc = self.lib.akshar_load_spm_model(self._h, bytes(data), len(data))
        if rc != 0:
            self._err(rc, 'akshar_load_spm_model')
        self._vocab.pop(1, None)
        self._pad.pop(1, None)

    def vocab(self, kind):
        """[(token str, type)] by id; kind 0 BPE, 1 Unigram"""
        if kind not in self._vocab:
            n = self.lib.akshar_vocab_size(self._h, kind)
            if n < 0:
                self._err(n, 'akshar_vocab_size')
            out = []
            p, ln, ty = ctypes.c_void_p(), ctypes.c_int(), ctypes.c_int()
            i = 0
            while True:
                rc = self.lib.akshar_vocab_token(self._h, kind, i, ctypes.byref(p), ctypes.byref(ln), ctypes.byref(ty))
                if rc != 0:
                    break
                raw = ctypes.string_at(p.value, ln.value) if ln.value else b''
                out.append((raw.decode('utf-8', errors='replace'), ty.value))
                i += 1
            self._vocab[kind] = (n, out)
        return self._vocab[kind]

    def _encode(self, fn, what, batch, mode, capacity, check):
        b = self.put(batch)
        cap = capacity if capacity is not None else (b.n_bytes >> 1) + 2 * b.n_rows + 1024
        ws = self._workspace(b.n_bytes, b.n_rows)
        word_extra = 0
        for _ in range(self.MAX_TRIES):
            ids = torch.empty(max(cap, 1), dtype=torch.int32, device=self.device)
            splits = torch.empty(b.n_rows + 1, dtype=torch.int64, device=self.device)
            result = torch.empty(4, dtype=torch.int64, device=self.device)
            rc = fn(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, b.begin, b.end, mode, ids.data_ptr(), cap,
                    splits.data_ptr(), result.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
            if rc != 0:
                self._err(rc, what)
            if not check:
                return Ragged(ids, splits), result
            total, _, bits = self._finish(result, what, True)
            if bits & C.ST_PATHOLOGICAL and mode == C.MODE_TILES:
                mode = C.MODE_ROWS
                continue
            if bits & C.ST_WORD and word_extra < 64:
                # a batch full of very long words ran out of the long-word pool: half of the workspace beyond the library's
                # minimum goes to that pool (include/akshar_b200.h), so grow the workspace and call again
                word_extra = 16 if word_extra == 0 else 64
                ws = self._workspace(b.n_bytes, b.n_rows, extra=word_extra * b.n_bytes + (4 << 20))
                continue
            if bits & C.ST_OVERFLOW:
                cap = max(cap, total)
                ws = self._workspace(b.n_bytes, b.n_rows, extra=max(ws.numel() - self.lib.akshar_workspace_bytes(b.n_bytes, b.n_rows), self._slot_extra(b.n_bytes)))
                continue
            if bits:
                raise BatchStatusError(bits, what)
            return Ragged(ids[:total], splits)
        raise BatchStatusError(bits, what + ' (retries exhausted)')

    def encode_bpe_batch(self, batch, mode=C.MODE_TILES, capacity=None, check=True):
        """Tokenizer.encode(norm).ids over ALREADY NORMALIZED rows (reference tokenizer.py:193) -> Ragged int32 ids"""
        return self._encode(self.lib.akshar_encode_bpe_batch, 'encode_bpe_batch', batch, mode, capacity, check)

    def encode_unigram_batch(self, batch, mode=C.MODE_TILES, capacity=None, check=True):
        """SentencePieceProcessor.EncodeAsIds(norm) over ALREADY NORMALIZED rows (reference tokenizer.py:191)"""
        return self._encode(self.lib.akshar_encode_unigram_batch, 'encode_unigram_batch', batch, mode, capacity, check)


    def tokenizer_encode_batch(self, batch, kind, normalize_roman=True, clean_hinglish=True, mode=C.MODE_TILES,
                               capacity=None, check=True):
        """aksharTokenizer.encode over RAW rows (reference tokenizer.py:167-193): normalize_text then the model, with no
        host synchronisation in between.  kind 0 BPE, 1 Unigram.  -> (ids Ragged, normalized TextBatch)"""
        b = self.put(batch)
        flags = (C.NORM_ROMAN if normalize_roman else 0) | (C.NORM_CLEAN if clean_hinglish else 0)
        ncap = b.n_bytes + (b.n_bytes >> 3) + 1024
        cap = capacity if capacity is not None else (b.n_bytes >> 1) + 2 * b.n_rows + 1024
        ws = self._workspace(ncap, b.n_rows)
        word_extra = 0
        for _ in range(self.MAX_TRIES):
            dev = self.device
            norm = torch.empty(max(ncap, 1), dtype=torch.uint8, device=dev)
            norm_off = torch.empty(b.n_rows + 1, dtype=torch.int64, device=dev)
            ids = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
            splits = torch.empty(b.n_rows + 1, dtype=torch.int64, device=dev)
            result = torch.empty(4, dtype=torch.int64, device=dev)
            rc = self.lib.akshar_tokenizer_encode_batch(self._h, b.data.data_ptr(), b.offsets.data_ptr(), b.n_rows, b.begin,
                                                        b.end, flags, kind, mode, norm.data_ptr(), ncap, norm_off.data_ptr(),
                                                        ids.data_ptr(), cap, splits.data_ptr(), result.data_ptr(),
                                                        ws.data_ptr(), ws.numel(), self._stream())
            if rc != 0:
                self._err(rc, 'akshar_tokenizer_encode_batch')
            if not check:
                return Ragged(ids, splits), TextBatch(norm, norm_off, 0, -1), result
            total, nbytes, bits = self._finish(result, 'tokenizer_encode', True)
            if bits & C.ST_PATHOLOGICAL and mode == C.MODE_TILES:
                mode = C.MODE_ROWS
                continue
            if bits & C.ST_WORD and word_extra < 64:
                word_extra = 16 if word_extra == 0 else 64         # long-word pool: see _encode
                ws = self._workspace(ncap, b.n_rows, extra=word_extra * b.n_bytes + (4 << 20))
                continue
            if bits & C.ST_OVERFLOW:
                # totals are exact even when a capacity was too small
                cap = max(cap, total)
                if nbytes > ncap:
                    ncap = nbytes
                    cap = max(cap, (ncap >> 1) + 2 * b.n_rows + 1024)
                ws = self._workspace(ncap, b.n_rows, extra=max(ws.numel() - self.lib.akshar_workspace_bytes(ncap, b.n_rows), self._slot_extra(ncap)))
                continue
            if bits:
                raise BatchStatusError(bits, 'tokenizer_encode_batch')
            return Ragged(ids[:total], splits), TextBatch(norm, norm_off, 0, nbytes)
        raise BatchStatusError(bits, 'tokenizer_encode_batch (retries exhausted)')


    # ------------------------------------------------------------------ host -> ids, pipelined
    def encode_host_pipelined(self, h_data, h_off, kind, normalize_roman=True, clean_hinglish=True, chunk_bytes=None,
                              out_ids=None, out_splits=None, compact=False):
        """aksharTokenizer.encode over a batch that lives in (pinned) HOST memory, returning host tensors: the batch is cut
        into row ranges of ~chunk_bytes; the H2D copy of chunk k+1, the kernels of chunk k and the D2H copy of chunk k-2
        run on three streams.

        compact=False -> (ids int32 [total], row_splits int64 [n_rows + 1])
        compact=True  -> `CompactIds`: uint16 ids (the vocabulary must fit) and int32 row splits RELATIVE TO THEIR CHUNK
                         (+ the chunks' first rows and first ids): a third of the bytes over the host link;
                         `.row_splits()` widens them on the host.

        Without out_ids / out_splits the results are views of pinned buffers that the engine keeps and REUSES: they are
        valid until the next call of this method on the same engine (pinning fresh memory for every call would cost more
        than the call).  A caller that needs them longer passes its own pinned tensors; a tensor that is too small is an
        error, it is never swapped silently."""
        import os
        import numpy as np
        from . import shard
        if chunk_bytes is None:
            # 64 MiB keeps both copy engines busy for BPE; the Unigram path has a latency floor per call (its exact-Viterbi
            # check walks whole rows), which 128 MiB chunks amortize (measured: 32 -> 40 GB/s end to end)
            chunk_bytes = int(os.environ.get('AKSHAR_CHUNK_MB', '64' if kind == 0 else '128')) << 20
        dev = self.device
        n_rows = h_off.numel() - 1
        off_np = h_off.numpy()
        total_bytes = int(off_np[-1] - off_np[0])
        ranges = shard.chunk_rows(off_np, chunk_bytes)
        max_b = max(int(off_np[hi] - off_np[lo]) for lo, hi in ranges)
        max_r = max(hi - lo for lo, hi in ranges)
        flags = (C.NORM_ROMAN if normalize_roman else 0) | (C.NORM_CLEAN if clean_hinglish else 0)
        if compact and self.lib.akshar_vocab_size(self._h, kind) > 65536:
            raise ValueError('compact ids need a vocabulary of at most 65536 entries')
        out_flags = (C.OUT_IDS_U16 | C.OUT_SPLITS_I32) if compact else 0
        id_dtype = torch.int16 if compact else torch.int32          # (uint16 bit patterns; torch copies them as they are)
        sp_dtype = torch.int32 if compact else torch.int64
        ncap = max_b + (max_b >> 3) + 1024
        cap = (max_b >> 1) + 2 * max_r + 1024
        ws = self._workspace(ncap, max_r)
        # pinned result buffers, device double buffers and streams are kept by the engine: repeated calls allocate nothing
        pc = self.__dict__.setdefault('_pipe_cache', {})
        est = (total_bytes >> 1) + 2 * n_rows + 1024
        key_sp, key_id = ('splits', sp_dtype), ('ids', id_dtype)
        if out_splits is None:
            if pc.get(key_sp) is None or pc[key_sp].numel() != n_rows + 1:
                pc[key_sp] = torch.empty(n_rows + 1, dtype=sp_dtype).pin_memory()
            out_splits = pc[key_sp]
        elif out_splits.numel() < n_rows + 1 or out_splits.dtype != sp_dtype:
            raise ValueError('out_splits must hold n_rows + 1 = %d entries of %s' % (n_rows + 1, sp_dtype))
        own_ids = out_ids is not None
        if out_ids is None:
            if pc.get(key_id) is None or pc[key_id].numel() < est:
                pc[key_id] = torch.empty(est, dtype=id_dtype).pin_memory()
            out_ids = pc[key_id]
        elif out_ids.dtype != id_dtype:
            raise ValueError('out_ids must be %s' % id_dtype)
        if 'streams' not in pc:
            pc['streams'] = tuple(torch.cuda.Stream(device=dev) for _ in range(3))
        s_in, s_comp, s_out = pc['streams']
        NSETS = 3        # input / compute / output of three consecutive chunks in flight; the host trails two chunks behind
        key = (max_b, max_r, NSETS, compact)
        sets = pc.get('sets') if pc.get('sets_key') == key else None
        if sets is None:
            sets = []
            for _ in range(NSETS):
                sets.append({
                    'text': torch.empty(max(max_b, 1), dtype=torch.uint8, device=dev),
                    'off': torch.empty(max_r + 1, dtype=torch.int64, device=dev),
                    'norm': torch.empty(max(ncap, 1), dtype=torch.uint8, device=dev),
                    'norm_off': torch.empty(max_r + 1, dtype=torch.int64, device=dev),
                    'ids': torch.empty(max(cap, 1), dtype=id_dtype, device=dev),
                    'splits': torch.empty(max_r + 1, dtype=sp_dtype, device=dev),
                    'result': torch.empty(4, dtype=torch.int64, device=dev),
                    'ev_in': torch.cuda.Event(), 'ev_comp': torch.cuda.Event(), 'ev_out': torch.cuda.Event(),
                })
        pc['sets'], pc['sets_key'] = sets, key
        cur = torch.cuda.current_stream(dev)
        for st in (s_in, s_comp, s_out):
            st.wait_stream(cur)
        state = {'tok': 0}
        chunk_rows = np.array([lo for lo, _ in ranges] + [n_rows], dtype=np.int64)
        chunk_ids = np.zeros(len(ranges) + 1, dtype=np.int64)
        trace = [] if os.environ.get('AKSHAR_PIPE_TRACE') else None
        if trace is not None:
            t0ev = torch.cuda.Event(enable_timing=True)
            t0ev.record(cur)

        def mark(stream, what, k):
            if trace is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record(stream)
                trace.append((what, k, e))

        def redo_chunk(k):
            """a chunk whose fast call raised a status: the same rows through the plain path (which retries with larger
            capacities / the row-by-row mode) -- only this chunk, the others keep their results"""
            lo, hi = ranges[k]
            b0, b1 = int(off_np[lo]), int(off_np[hi])
            sub = (h_data[b0:b1], (h_off[lo:hi + 1] - b0))
            with torch.cuda.stream(s_out):
                ids, _ = self.tokenizer_encode_batch(sub, kind, normalize_roman, clean_hinglish)
                v = ids.values
                sp = ids.splits
                if compact:
                    v = v.to(torch.int16)
                    sp = sp.to(torch.int32)
                return v, sp, int(v.numel())

        def finish(k):
            lo, hi = ranges[k]
            S = sets[k % NSETS]
            with torch.cuda.stream(s_out):
                s_out.wait_event(S['ev_comp'])
                r = S['result'].cpu()          # waits for chunk k's kernels only; later chunks are already enqueued
                n, bits = int(r[0]), int(r[2])
                d_ids, d_sp = S['ids'], S['splits']
                if bits:
                    self.redone_chunks = getattr(self, 'redone_chunks', 0) + 1
                    d_ids, d_sp, n = redo_chunk(k)
                if state['tok'] + n > out_ids.numel():
                    if own_ids:
                        raise ValueError('out_ids is too small: %d ids so far, %d more in this chunk' % (state['tok'], n))
                    grown = torch.empty(max(2 * out_ids.numel(), state['tok'] + n), dtype=id_dtype).pin_memory()
                    torch.cuda.synchronize(dev)
                    grown[:state['tok']].copy_(out_ids[:state['tok']])
                    pc[key_id] = grown
                    state['out_ids'] = grown
                dst = state.get('out_ids', out_ids)
                mark(s_out, 'd2h_begin', k)
                dst[state['tok']:state['tok'] + n].copy_(d_ids[:n], non_blocking=True)
                sp = d_sp[1:hi - lo + 1]
                if not compact and state['tok']:
                    sp = sp + state['tok']
                out_splits[lo + 1:hi + 1].copy_(sp, non_blocking=True)
                S['ev_out'].record(s_out)
                mark(s_out, 'd2h_end', k)
                chunk_ids[k] = state['tok']
                state['tok'] += n

        out_splits[0] = 0
        try:
            for k, (lo, hi) in enumerate(ranges):
                S = sets[k % NSETS]
                b0, b1 = int(off_np[lo]), int(off_np[hi])
                nb, nr = b1 - b0, hi - lo
                with torch.cuda.stream(s_in):
                    if k >= NSETS:
                        s_in.wait_event(S['ev_comp'])      # the kernels that read this input buffer have finished
                    # the rows keep their ABSOLUTE offsets (the C ABI takes text_begin / text_end): no per-chunk rebasing on
                    # the host, the offsets go to the device straight from the caller's (pinned) array
                    mark(s_in, 'h2d_begin', k)
                    S['text'][:nb].copy_(h_data[b0:b1], non_blocking=True)
                    S['off'][:nr + 1].copy_(h_off[lo:hi + 1], non_blocking=True)
                    S['ev_in'].record(s_in)
                    mark(s_in, 'h2d_end', k)
                with torch.cuda.stream(s_comp):
                    s_comp.wait_event(S['ev_in'])
                    if k >= NSETS:
                        s_comp.wait_event(S['ev_out'])     # chunk k-NSETS's results left this set's output buffers
                    rc = self.lib.akshar_tokenizer_encode_batch_ex(
                        self._h, S['text'].data_ptr() - b0, S['off'].data_ptr(), nr, b0, b1, flags, kind, C.MODE_TILES,
                        S['norm'].data_ptr(), ncap, S['norm_off'].data_ptr(), S['ids'].data_ptr(), cap, S['splits'].data_ptr(),
                        out_flags, S['result'].data_ptr(), ws.data_ptr(), ws.numel(), ctypes.c_void_p(s_comp.cuda_stream))
                    if rc != 0:
                        self._err(rc, 'akshar_tokenizer_encode_batch_ex')
                    S['ev_comp'].record(s_comp)
                    mark(s_comp, 'comp_end', k)
                if k >= 2:
                    finish(k - 2)          # its kernels ended while chunk k-1 ran: no wait, the copy engines never idle
            for k in range(max(0, len(ranges) - 2), len(ranges)):
                finish(k)
        finally:
            for st in (s_in, s_comp, s_out):
                cur.wait_stream(st)
            torch.cuda.synchronize(dev)
        if trace:
            print('pipe trace (ms): ' + ' '.join('%s%d=%.2f' % (w, k, t0ev.elapsed_time(e)) for w, k, e in trace))
        out_ids = state.get('out_ids', out_ids)
        chunk_ids[len(ranges)] = state['tok']
        if compact:
            return CompactIds(out_ids[:state['tok']], out_splits[:n_rows + 1], chunk_rows, chunk_ids)
        return out_ids[:state['tok']], out_splits[:n_rows + 1]


class PipelineOut:
    """normalize -> akshars -> script runs of a batch as it crosses the host link (Engine.pipeline_host_pipelined): the
    normalized rows (bytes + int64 row offsets) and, per chunk of rows, the boundary bit masks of AKSHAR_SEG_MASK.  Chunk c
    holds rows chunk_rows[c] .. chunk_rows[c + 1] - 1; its text starts at norm byte chunk_bytes[c] and its mask words at
    chunk_words[c] (bit i of the chunk's mask = byte chunk_bytes[c] + i)."""

    def __init__(self, norm, offsets, cmask, rmask, t0, t1, chunk_rows, chunk_bytes, chunk_words, n_clusters, n_runs):
        self.norm, self.offsets = norm, offsets
        self.cmask, self.rmask, self.t0, self.t1 = cmask, rmask, t0, t1
        self.chunk_rows, self.chunk_bytes, self.chunk_words = chunk_rows, chunk_bytes, chunk_words
        self.n_clusters, self.n_runs = n_clusters, n_runs

    def _ends(self, mask):
        """absolute byte positions (in `norm`) of the set bits, ascending"""
        import numpy as np
        out = []
        for c in range(len(self.chunk_rows) - 1):
            w = mask[self.chunk_words[c]:self.chunk_words[c + 1]].numpy().view(np.uint32)
            bits = np.unpackbits(w.view(np.uint8), bitorder='little')
            out.append(np.flatnonzero(bits) + self.chunk_bytes[c])
        return np.concatenate(out) if out else np.zeros(0, dtype=np.int64)

    def cluster_ends(self):
        """-> (int32 END offsets relative to the row start, int64 row splits): the form segment_batch returns"""
        return self._ragged(self._ends(self.cmask))

    def run_ends(self):
        """-> (ends, splits, uint8 tags)"""
        import numpy as np
        pos = self._ends(self.rmask)
        b0 = np.isin(pos, self._ends(self.t0), assume_unique=True)
        b1 = np.isin(pos, self._ends(self.t1), assume_unique=True)
        tags = np.where(b0 & b1, 255, np.where(b0, 1, np.where(b1, 4, 0))).astype(np.uint8)
        e, sp = self._ragged(pos)
        return e, sp, tags

    def _ragged(self, pos):
        import numpy as np
        off = self.offsets.numpy()
        # an end at position p belongs to the row with off[r] < p <= off[r + 1]
        row = np.searchsorted(off, pos, side='left') - 1
        splits = np.searchsorted(row, np.arange(off.size), side='left').astype(np.int64)
        return (pos - off[row]).astype(np.int32), splits


class CompactIds:
    """ids of a batch as they cross the host link: uint16 ids (held in an int16 tensor, same bits) and int32 row splits
    relative to the first id of the row's CHUNK; chunk c holds rows chunk_rows[c] .. chunk_rows[c + 1] - 1 and its first
    id is ids[chunk_ids[c]]"""

    def __init__(self, ids, splits32, chunk_rows, chunk_ids):
        self.ids16 = ids
        self.splits32 = splits32
        self.chunk_rows = chunk_rows
        self.chunk_ids = chunk_ids

    def numel(self):
        return self.ids16.numel()

    def ids(self):
        """uint16 numpy view of the ids"""
        import numpy as np
        return self.ids16.numpy().view(np.uint16)

    def row_splits(self):
        """int64 row splits of the whole batch (widened on the host)"""
        import numpy as np
        sp = self.splits32.numpy().astype(np.int64)
        for c in range(len(self.chunk_rows) - 1):
            lo, hi = int(self.chunk_rows[c]), int(self.chunk_rows[c + 1])
            sp[lo + 1:hi + 1] += int(self.chunk_ids[c])
        sp[0] = 0
        return sp


_engines = {}


def engine(device=0):
    """process-wide engine per device"""
    if device not in _engines:
        _engines[device] = Engine(device)
    return _engines[device]
