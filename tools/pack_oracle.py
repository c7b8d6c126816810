"""Packed language-model batches in plain Python (no torch, no transformers): the rule of Engine.pack_batch and of
akshar_pack_count / akshar_pack_write (include/akshar_b200.h).

1. Stream: the carry's fragments verbatim, then every row's ids, each followed by `eos_id` when one is given.  A
   document start is the start of a non-empty fragment or row.
2. Blocks: T = |S|, N = T // L; block b is S[b L : (b + 1) L] (transformers' run_clm.py `group_texts`).  The remainder
   S[N L : T] (< L ids) is returned as `rest`, its document starts as fragment splits; passing it as the next call's
   carry makes packing in chunks equal packing in one call.
3. Pieces start at every block start and at every document start below N L; the outputs are what transformers'
   DataCollatorWithFlattening returns for the list of pieces in order.
"""


def stream(rows, eos_id=None, carry=None):
    """-> (S, document starts): the ids of the call in stream order and the starts of its non-empty units"""
    S, starts = [], []
    units = []
    if carry is not None:
        values, splits = carry
        units += [list(values[splits[i]:splits[i + 1]]) for i in range(len(splits) - 1)]
    units += [list(r) + ([eos_id] if eos_id is not None else []) for r in rows]
    for u in units:
        if u:
            starts.append(len(S))
            S.extend(u)
    return S, starts


def group_texts(ids, block_size):
    """run_clm.py's group_texts over one concatenated stream: whole blocks only, the remainder dropped"""
    total = len(ids) // block_size * block_size
    return [ids[i:i + block_size] for i in range(0, total, block_size)]


def piece_starts(T, starts, block_size):
    NL = T // block_size * block_size
    return sorted(set(range(0, NL, block_size)) | {d for d in starts if d < NL}), NL


def pack(rows, block_size, eos_id=None, carry=None, separator_id=-100):
    """-> (pieces, rest): the pieces in order (lists of ids) and rest = (values, splits)"""
    if block_size < 1:
        raise ValueError('block_size must be at least 1')
    S, starts = stream(rows, eos_id, carry)
    T = len(S)
    ps, NL = piece_starts(T, starts, block_size)
    pieces = [S[a:b] for a, b in zip(ps, ps[1:] + [NL])]
    rest_splits = [0] + [d - NL for d in starts if NL < d < T] + ([T - NL] if T > NL else [])
    return pieces, (S[NL:], rest_splits)


def flatten(pieces, separator_id=-100):
    """DataCollatorWithFlattening(return_flash_attn_kwargs=True, return_seq_idx=True) over the pieces, as flat lists"""
    out = {'input_ids': [], 'labels': [], 'position_ids': [], 'seq_idx': []}
    cu, longest = [0], 0
    for k, p in enumerate(pieces):
        out['input_ids'] += p
        out['labels'] += [separator_id] + p[1:]
        out['position_ids'] += list(range(len(p)))
        out['seq_idx'] += [k] * len(p)
        cu.append(cu[-1] + len(p))
        longest = max(longest, len(p))
    out['cu_seq_lens'] = cu
    out['max_length'] = longest
    return out


def unit_pieces(s, length, block_size, NL):
    """closed form of one unit (fragment or row) at stream start s: (pieces that start in it below NL, longest of them,
    rest fragments that start in it)"""
    L = block_size
    e = s + length
    if length <= 0:
        return 0, 0, 0
    rest = 1 if e > NL else 0
    if s >= NL:
        return 0, 0, rest
    m = min(e, NL)
    n = 1 + (m - 1) // L - s // L
    first = min(m, (s // L + 1) * L) - s
    longest = first
    if n >= 2:
        longest = max(longest, m - (m - 1) // L * L)
    if n >= 3:
        longest = L
    return n, longest, rest


def position(p, s, k, block_size):
    """(position_ids[p], seq_idx[p]) of a position p < NL in the unit at stream start s whose first piece is piece k"""
    b = p // block_size
    return p - max(s, b * block_size), k + b - s // block_size
