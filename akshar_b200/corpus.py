"""File / corpus front end of the hot path (SURVEY.md section 8f-1): the callers on either side of the batch kernels.

Mirrors, on the batch path, what the reference does one string at a time:
  * `preprocess_corpus`  = reference cli.py:165-190 (= scripts/train_bpe.py:16-35, train_spm.py:18-44): read lines,
    `strip()`, skip the empty ones, `normalize_text` each, write them back one per line;
  * `tokenize_file`      = reference cli.py:46-84 `akshar tokenize -i FILE --format text|json|id`: the WHOLE file is one
    string (one very long row for the kernels);
  * `encode_lines`       = new: one row per non-empty line, ragged ids back.

No Python work per line: the file is read in large pieces straight into pinned host memory (`readinto`), each piece is cut
at its last line terminator, copied to the device while the previous piece is being processed, and split into stripped,
non-empty rows there (Engine.lines_batch -> akshar_lines_batch).  The bytes must be valid UTF-8 (Python's text-mode
`open` would raise UnicodeDecodeError otherwise; the device path does not check).
"""
import json

import numpy as np
import torch

from .batch import engine

CHUNK_BYTES = 256 << 20


class _PinnedPieces:
    """pieces of a file, each ending at a line terminator (or at the end of the file), in two pinned buffers used in turn"""

    def __init__(self, path, chunk_bytes):
        self.f = open(path, 'rb', buffering=0)
        self.cap = max(int(chunk_bytes), 1 << 16)
        self.bufs = [torch.empty(self.cap, dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.turn = 0
        self.carry = np.zeros(0, dtype=np.uint8)
        self.eof = False

    def close(self):
        self.f.close()

    def _grow(self, need):
        cap = self.cap
        while cap < need:
            cap *= 2
        if cap != self.cap:
            self.cap = cap
            self.bufs = [torch.empty(cap, dtype=torch.uint8).pin_memory() for _ in range(2)]

    def next(self):
        """-> (pinned uint8 tensor, n_bytes) or None"""
        while True:
            if self.eof and self.carry.size == 0:
                return None
            self._grow(self.carry.size + (1 << 16))
            buf = self.bufs[self.turn]
            view = buf.numpy()
            have = self.carry.size
            view[:have] = self.carry
            while have < self.cap and not self.eof:
                got = self.f.readinto(memoryview(view)[have:self.cap])
                if not got:
                    self.eof = True
                    break
                have += got
            if self.eof:
                self.carry = np.zeros(0, dtype=np.uint8)
                self.turn ^= 1
                return buf, have
            # cut after the last '\n' / '\r' of the piece; what follows waits for the next one
            cut = -1
            hi = have
            while hi > 0 and cut < 0:
                lo = max(0, hi - (1 << 20))
                w = view[lo:hi]
                idx = np.flatnonzero((w == 10) | (w == 13))
                if idx.size:
                    cut = lo + int(idx[-1]) + 1
                hi = lo
            if cut < 0:
                # one line longer than the buffer: take a bigger one and read on
                self.carry = view[:have].copy()
                self._grow(2 * self.cap)
                continue
            self.carry = view[cut:have].copy()
            self.turn ^= 1
            return buf, cut


def stream_rows(input_file, device=0, chunk_bytes=CHUNK_BYTES):
    """generator of device TextBatch objects: the stripped, non-empty lines of the file, one piece at a time; the host
    read + copy of piece k + 1 overlaps the device work on piece k (the consumer's)"""
    eng = engine(device)
    pieces = _PinnedPieces(input_file, chunk_bytes)
    copy_stream = torch.cuda.Stream(device=eng.device)
    try:
        nxt = pieces.next()
        staged = None
        if nxt is not None:
            staged = _stage(eng, copy_stream, nxt)
        while staged is not None:
            d_file, n, ev = staged
            nxt = pieces.next()                      # host read of the next piece while the copy of this one runs
            torch.cuda.current_stream(eng.device).wait_event(ev)
            rows = eng.lines_batch(d_file, n)
            staged = _stage(eng, copy_stream, nxt) if nxt is not None else None
            yield rows
    finally:
        pieces.close()


def _stage(eng, stream, piece):
    buf, n = piece
    d = torch.empty(max(n, 1) + 8, dtype=torch.uint8, device=eng.device)
    with torch.cuda.stream(stream):
        d[:n].copy_(buf[:n], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(stream)
    d.record_stream(torch.cuda.current_stream(eng.device))
    return d, n, ev


def read_rows(input_file, device=0):
    """the reference's row definition (readlines / strip / skip empty), computed on the device -> list[str]"""
    out = []
    for rows in stream_rows(input_file, device):
        out.extend(rows.to_strings())
    return out


def preprocess_corpus(input_file, output_file, normalize_roman=True, clean_hinglish=True, device=0, chunk_bytes=CHUNK_BYTES):
    """reference cli.py:165-190: file -> normalized lines, one per line.  disk -> pinned -> device -> rows -> normalize_text
    -> rows joined by '\\n' on the device -> disk"""
    print(f"Preprocessing {input_file}...")
    eng = engine(device)
    n_lines = 0
    with open(output_file, 'wb') as out:
        for rows in stream_rows(input_file, device, chunk_bytes):
            if rows.n_rows == 0:
                continue
            norm = eng.normalize_batch(rows, normalize_roman, clean_hinglish)
            out.write(eng.join_rows(norm).cpu().numpy().tobytes())
            n_lines += norm.n_rows
    print(f"Wrote {n_lines} lines to {output_file}")
    return str(output_file)


def _whole_file(input_file):
    """the file as ONE string, as the reference's `f.read()` of a text-mode file gives it (universal newlines)"""
    with open(input_file, 'rb') as f:
        data = f.read()
    if b'\r' in data:
        data = data.replace(b'\r\n', b'\n').replace(b'\r', b'\n')
    return data


def tokenize_file(tokenizer, input_file, fmt='text', output_file=None):
    """-> the string the reference CLI would print / write (cli.py:46-84)"""
    data = _whole_file(input_file)
    arr = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()) if data else torch.zeros(0, dtype=torch.uint8)
    batch = (arr, torch.tensor([0, len(data)], dtype=torch.int64))
    if fmt == 'id':
        if tokenizer.model is None:
            raise ValueError("need model for IDs")
        output = ' '.join(map(str, tokenizer.encode_batch(batch)[0]))
    else:
        tokens = tokenizer.tokenize_batch(batch)[0]
        output = json.dumps(tokens, ensure_ascii=False, indent=2) if fmt == 'json' else ' '.join(tokens)
    if output_file:
        with open(output_file, 'w', encoding='utf-8') as f:
            f.write(output)
    return output


def encode_lines(tokenizer, input_file, as_device=False, chunk_bytes=CHUNK_BYTES):
    """one row per non-empty stripped line -> list[list[int]] (or, with as_device=True, a list of device Ragged objects,
    one per piece of the file)"""
    if tokenizer.model is None:
        raise ValueError("need model for IDs")
    out = []
    for rows in stream_rows(input_file, tokenizer._device, chunk_bytes):
        ids, _ = tokenizer.encode_batch(rows, as_device=True)
        if as_device:
            out.append(ids)
        else:
            out.extend(r.tolist() for r in ids.rows())
    return out


def pack_lines(tokenizer, input_file, block_size, chunk_bytes=CHUNK_BYTES, mlm=None, **kwargs):
    """generator of packed causal-LM batches of a text file, one per piece of the file: every non-empty stripped line is
    a document, encoded on the device and packed by Engine.pack_batch (keywords: eos_id, separator_id,
    return_position_ids, return_seq_idx, return_flash_attn_kwargs).  The rest of each piece is the carry of the next,
    so the blocks are those of packing the whole file in one call.  The ids after the file's last whole block are
    dropped, as transformers' run_clm.py `group_texts` drops them.
    mlm: a dict of Engine.mlm_mask keywords (seed, mlm_probability, mask_replace_prob, random_replace_prob, epoch,
    mask_id, pad_id); every batch is then masked for masked-LM training, its labels replaced by the masked-LM ones, with
    row_base = the blocks yielded before it, so that the masks are those of masking the one-call batch."""
    if tokenizer.model is None:
        raise ValueError("need model for IDs")
    if 'carry' in kwargs:
        raise ValueError('pack_lines threads the carry itself')
    if mlm is not None and (not isinstance(mlm, dict) or 'row_base' in mlm):
        raise ValueError('mlm must be a dict of mlm_mask keywords without row_base: pack_lines threads the row_base itself')
    carry = None
    row_base = 0
    for rows in stream_rows(input_file, tokenizer._device, chunk_bytes):
        ids, _ = tokenizer.encode_batch(rows, as_device=True)
        batch, carry = tokenizer._eng.pack_batch(ids, block_size, carry=carry, **kwargs)
        if mlm is not None:
            batch['labels'] = tokenizer._eng.mlm_mask(batch['input_ids'], tokenizer.model.kind, row_base=row_base, **mlm)[1]
            row_base += batch['input_ids'].shape[0]
        yield batch
