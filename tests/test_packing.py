"""Packed language-model batches (fixed blocks with per-document position_ids, labels, seq_idx and cu_seq_lens): the
oracle (tools/pack_oracle.py) against what transformers' DataCollatorWithFlattening returned
(tests/golden/packing_hf.json.gz, tools/make_golden_packing.py), the AK_HD arithmetic of the kernels (ak_pack.cuh, built
on the CPU with tests/csrc/pack_shim.cpp) against the oracle, and the device path (Engine.pack_batch,
aksharTokenizer.encode_batch_packed, corpus.pack_lines) against both."""
import ctypes
import gzip
import json
import os
import random
import subprocess
import zlib

import numpy as np
import pytest

import pack_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
MODELS = os.path.join(GOLDEN, 'models')
KEYS = ('input_ids', 'labels', 'position_ids', 'seq_idx')


@pytest.fixture(scope='module')
def fix():
    with gzip.open(os.path.join(GOLDEN, 'packing_hf.json.gz'), 'rb') as f:
        return json.loads(f.read().decode('utf-8'))


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


def oracle_summary(pieces, rest, L):
    """the fixture's record of one call, from the oracle's pieces and rest"""
    flat = O.flatten(pieces)
    cu = flat['cu_seq_lens']
    return {'N': sum(len(p) for p in pieces) // L, 'pieces': [b - a for a, b in zip(cu, cu[1:])],
            'max_length': flat['max_length'], 'rest': [b - a for a, b in zip(rest[1], rest[1][1:])],
            'rest_crc': crc(np.asarray(rest[0], np.int32)),
            'crc': {'input_ids': crc(np.asarray(flat['input_ids'], np.int64)), 'labels': crc(np.asarray(flat['labels'], np.int64)),
                    'position_ids': crc(np.asarray(flat['position_ids'], np.int64)),
                    'seq_idx': crc(np.asarray(flat['seq_idx'], np.int32)), 'cu_seq_lens_q': crc(np.asarray(cu, np.int32))}}


def strip(rec):
    return {k: v for k, v in rec.items() if not k.startswith('verbatim')}


def configurations(fix, golden):
    """(source name, eos, batch index, L, [(rows, carry) per call], [fixture record per call]) for every one-call and
    chained configuration"""
    rows = golden['rows']
    for name, src in fix['sources'].items():
        for bi, b in enumerate(fix['batches']):
            ids = [rows[i][src['key']] for i in b]
            c1, c2 = fix['cuts'][bi]
            for L in fix['block_sizes']:
                yield name, src['eos'], bi, L, [ids], [src['one'][bi][str(L)]]
                yield name, src['eos'], bi, L, [ids[:c1], ids[c1:c2], ids[c2:]], src['chain'][bi][str(L)]


# ------------------------------------------------------------------ CPU: the oracle is the collator
def test_fixture_holds_every_configuration(fix):
    assert fix['pins'] == {'transformers': '5.5.0'}
    assert fix['block_sizes'] == [1, 2, 3, 8, 17, 64, 128, 512, 4096]
    assert len(fix['batches']) == 9 and all(len(b) == 64 for b in fix['batches'][:8]) and len(fix['batches'][8]) == 66
    assert set(fix['sources']) == {'bpe24k', 'spm24k', 'spm24k_eos'}
    assert fix['sources']['spm24k_eos']['eos'] == 2 and fix['sources']['bpe24k']['eos'] is None
    for src in fix['sources'].values():
        assert len(src['one']) == len(src['chain']) == 9
        assert all(len(c[str(L)]) == 3 for c in src['chain'] for L in fix['block_sizes'])


def test_fixture_batches_hold_the_edge_rows(fix, golden):
    rows = golden['rows']
    last = fix['batches'][8]
    assert len(rows[last[0]]['ids_bpe24k']) == 3558
    assert sum(1 for i in last if not rows[i]['ids_spm24k']) == 65


def test_oracle_equals_collator(fix, golden):
    """every configuration: N, piece lengths, max_length, the rest, and the CRC32 of every array the collator returned"""
    n = 0
    for name, eos, bi, L, calls, recs in configurations(fix, golden):
        carry = None
        for part, rec in zip(calls, recs):
            pieces, carry = O.pack(part, L, eos, carry)
            assert oracle_summary(pieces, carry, L) == strip(rec), (name, bi, L)
            n += 1
    assert n == 3 * 9 * 9 * 4


def test_oracle_equals_collator_verbatim(fix, golden):
    """the calls stored verbatim: every array, max_length and the rest, as the collator returned them"""
    seen = 0
    for name, eos, bi, L, calls, recs in configurations(fix, golden):
        carry = None
        for part, rec in zip(calls, recs):
            pieces, carry = O.pack(part, L, eos, carry)
            if 'verbatim' not in rec:
                continue
            flat = O.flatten(pieces)
            v = rec['verbatim']
            for key in KEYS:
                assert v[key] == [flat[key]], (name, bi, L, key)
            assert v['cu_seq_lens_q'] == v['cu_seq_lens_k'] == flat['cu_seq_lens']
            assert v['max_length_q'] == v['max_length_k'] == flat['max_length']
            assert rec['verbatim_rest'] == [list(carry[0]), list(carry[1])]
            seen += 1
    assert seen == 4                                    # one call, and the three calls of one chain


def test_oracle_is_group_texts():
    rows = [[5, 6, 7], [], [8], [9, 10, 11, 12, 13]]
    S, starts = O.stream(rows, 2)
    assert S == [5, 6, 7, 2, 2, 8, 2, 9, 10, 11, 12, 13, 2] and starts == [0, 4, 5, 7]
    pieces, rest = O.pack(rows, 4, 2)
    assert pieces == [[5, 6, 7, 2], [2], [8, 2], [9], [10, 11, 12, 13]]
    assert rest == ([2], [0, 1])
    assert [x for p in pieces for x in p] == [x for b in O.group_texts(S, 4) for x in b]
    assert O.pack(rows, 4, None) == ([[5, 6, 7], [8], [9, 10, 11, 12]], ([13], [0, 1]))
    assert O.pack([[1, 2]], 3) == ([], ([1, 2], [0, 2]))
    assert O.pack([], 3) == ([], ([], [0]))
    with pytest.raises(ValueError):
        O.pack(rows, 0)


# ------------------------------------------------------------------ CPU: the kernels' arithmetic is the oracle
@pytest.fixture(scope='module')
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp('pack_shim') / 'libpack_shim.so')
    subprocess.check_call(['g++', '-O1', '-std=c++17', '-shared', '-fPIC', '-o', so, os.path.join(ROOT, 'tests', 'csrc', 'pack_shim.cpp')])
    lib = ctypes.CDLL(so)
    vp, i64 = ctypes.c_void_p, ctypes.c_int64
    lib.ps_pack_units.argtypes = [vp, i64, i64, i64, vp]
    lib.ps_pack_positions.argtypes = [vp, i64, vp, i64, i64, vp, vp]
    lib.ps_pack_position.argtypes = [i64, i64, i64, i64, vp, vp]
    return lib


def unit_starts(parts_lens, eos, carry_lens):
    """stream starts of the units of a call (carry fragments, then rows with their eos), and T"""
    lens = list(carry_lens) + [n + (eos is not None) for n in parts_lens]
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int64) if lens else np.zeros(1, np.int64)


def shim_summary(shim, starts, L):
    """the record of one call from the shim's unit counts and positions (no ids: the id CRCs are left out)"""
    n_units, T = starts.size - 1, int(starts[-1])
    NL = T // L * L
    U = np.zeros((max(n_units, 1), 3), np.int64)
    shim.ps_pack_units(starts.ctypes.data, n_units, L, NL, U.ctypes.data)
    U = U[:n_units]
    first = np.concatenate([[0], np.cumsum(U[:, 0])]).astype(np.int64)
    pos = np.zeros(max(NL, 1), np.int32)
    seq = np.zeros(max(NL, 1), np.int32)
    shim.ps_pack_positions(starts.ctypes.data, n_units, first.ctypes.data, L, NL, pos.ctypes.data, seq.ctypes.data)
    pos, seq = pos[:NL], seq[:NL]
    ps = np.flatnonzero(pos == 0)
    assert ps.size == int(first[-1]) and np.array_equal(seq[ps], np.arange(ps.size))
    cu = np.append(ps, NL).astype(np.int32)
    rs = [NL] + [int(s) for s, e in zip(starts[:-1], starts[1:]) if NL < s < T and e > s] if T > NL else []
    assert len(rs) == int(U[:, 2].sum())
    return {'N': NL // L, 'pieces': np.diff(cu).tolist(), 'max_length': int(U[:, 1].max()) if n_units else 0,
            'rest': np.diff(rs + [T] if rs else [0]).tolist() if rs else [],
            'position_ids': crc(pos.astype(np.int64)), 'seq_idx': crc(seq), 'cu_seq_lens_q': crc(cu)}


def test_shim_equals_oracle_on_the_fixture(fix, golden, shim):
    for name, eos, bi, L, calls, recs in configurations(fix, golden):
        carry_lens = []
        carry = None
        for part, rec in zip(calls, recs):
            got = shim_summary(shim, unit_starts([len(r) for r in part], eos, carry_lens), L)
            want = {k: rec[k] for k in ('N', 'pieces', 'max_length', 'rest')}
            want.update({k: rec['crc'][k] for k in ('position_ids', 'seq_idx', 'cu_seq_lens_q')})
            assert got == want, (name, bi, L)
            _, carry = O.pack(part, L, eos, carry)
            carry_lens = np.diff(carry[1]).tolist()


def test_shim_near_2_31_equals_oracle(shim):
    """seeded units (s, len) that end just below 2^31, block sizes from 1 to 2^30: counts, longest piece and the
    position / piece index of sampled positions against the oracle's enumeration of the unit's pieces"""
    rng = random.Random(20261021)
    for _ in range(3000):
        L = rng.choice([1, 2, 3, 17, 64, 4096, 8192, 65536, 1 << 20, (1 << 30) + 7, rng.randint(1, 1 << 16)])
        T = (1 << 31) - 1 - rng.randint(0, 3 * L if L < (1 << 20) else 5)
        NL = T // L * L
        n = rng.randint(1, 3000 if L < 64 else 100000)
        s = max(0, T - n - rng.randint(0, 2 * L if L < 4096 else 9000))
        e = min(s + n, T)
        U = np.zeros(3, np.int64)
        st = np.array([s, e], np.int64)
        shim.ps_pack_units(st.ctypes.data, 1, L, NL, U.ctypes.data)
        want = O.unit_pieces(s, e - s, L, NL)
        # the oracle's enumeration: pieces of [s, min(e, NL)) at s and the block starts
        m = min(e, NL)
        starts = ([s] + list(range((s // L + 1) * L, m, L))) if s < NL else []
        lens = [b - a for a, b in zip(starts, starts[1:] + [m])]
        assert tuple(U) == want == (len(starts), max(lens, default=0), int(e > NL)), (s, e, L)
        k = rng.randint(0, 1 << 20)
        for i in rng.sample(range(len(starts)), min(len(starts), 4)):
            p = rng.randint(starts[i], starts[i] + lens[i] - 1)
            pos, seq = ctypes.c_int32(), ctypes.c_int32()
            shim.ps_pack_position(p, s, L, k, ctypes.byref(pos), ctypes.byref(seq))
            assert (pos.value, seq.value) == (p - starts[i], k + i) == O.position(p, s, k, L)


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope='module')
def A():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import __graft_entry__ as g
    g.build()
    import akshar_b200
    return akshar_b200


@pytest.fixture(scope='module')
def toks(A):
    return {'bpe24k': A.aksharTokenizer(os.path.join(MODELS, 'bpe24k.json'), 'bpe'),
            'spm24k': A.aksharTokenizer(os.path.join(MODELS, 'spm24k.model'), 'sentencepiece')}


ALL = dict(return_position_ids=True, return_seq_idx=True, return_flash_attn_kwargs=True)


def device_summary(batch, rest, L):
    """the fixture's record of one call, from the device outputs (checks their dtypes and shapes on the way)"""
    import torch
    n = batch['input_ids'].shape[0]
    for k in KEYS:
        t = batch[k]
        assert t.dtype == (torch.int32 if k == 'seq_idx' else torch.int64) and tuple(t.shape) == (n, L), k
    cu = batch['cu_seq_lens_q']
    assert cu.dtype == torch.int32 and torch.equal(cu, batch['cu_seq_lens_k'])
    assert isinstance(batch['max_length_q'], int) and batch['max_length_q'] == batch['max_length_k']
    assert list(batch) == ['input_ids', 'labels', 'position_ids', 'seq_idx', 'cu_seq_lens_q', 'cu_seq_lens_k', 'max_length_q',
                           'max_length_k']
    assert rest.values.dtype == torch.int32 and rest.splits.dtype == torch.int64
    cu_np = cu.cpu().numpy()
    rs = rest.splits.cpu().numpy()
    return {'N': n, 'pieces': np.diff(cu_np).tolist(), 'max_length': batch['max_length_q'], 'rest': np.diff(rs).tolist(),
            'rest_crc': crc(rest.values.cpu().numpy()),
            'crc': {k: crc(batch[k].cpu().numpy()) for k in KEYS + ('cu_seq_lens_q',)}}


def ragged_of(torch, rows, dtype, device):
    lens = np.array([len(r) for r in rows], dtype=np.int64)
    v = np.concatenate([np.asarray(r, np.int64) for r in rows]) if rows and lens.sum() else np.zeros(0, np.int64)
    v = torch.from_numpy(v.astype(np.uint16).view(np.int16) if dtype == 'uint16' else v.astype(np.int32))
    return v.to(device), torch.from_numpy(np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)).to(device)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', ['int32', 'uint16'])
@pytest.mark.parametrize('source', ['bpe24k', 'spm24k', 'spm24k_eos'])
def test_pack_batch_equals_fixture(A, fix, golden, toks, source, dtype):
    """Engine.pack_batch on the encoder's output of the golden rows' `in` strings, every batch and block size, in one
    call and as the fixture's 3-call carry chain"""
    import torch
    src = fix['sources'][source]
    tk = toks[source[:6]]
    eng = tk._eng
    rows = golden['rows']
    for bi, b in enumerate(fix['batches']):
        enc, _ = tk.encode_batch([rows[i]['in'] for i in b], as_device=True)
        got_rows = [r.tolist() for r in enc.rows()]
        assert got_rows == [rows[i][src['key']] for i in b]
        v, sp = ragged_of(torch, got_rows, dtype, eng.device)
        c1, c2 = fix['cuts'][bi]
        for L in fix['block_sizes']:
            batch, rest = eng.pack_batch((v, sp), L, eos_id=src['eos'], **ALL)
            assert device_summary(batch, rest, L) == strip(src['one'][bi][str(L)]), (bi, L)
            carry = None
            for (lo, hi), rec in zip(((0, c1), (c1, c2), (c2, len(b))), src['chain'][bi][str(L)]):
                batch, carry = eng.pack_batch((v, sp[lo:hi + 1]), L, eos_id=src['eos'], carry=carry, **ALL)
                assert device_summary(batch, carry, L) == strip(rec), (bi, L, lo)


@pytest.mark.gpu
@pytest.mark.parametrize('source', ['bpe24k', 'spm24k', 'spm24k_eos'])
def test_encode_batch_packed_equals_fixture(A, fix, golden, toks, source):
    src = fix['sources'][source]
    tk = toks[source[:6]]
    rows = golden['rows']
    for bi, b in enumerate(fix['batches']):
        texts = [rows[i]['in'] for i in b]
        c1, c2 = fix['cuts'][bi]
        for L in (1, 17, 512):
            batch, rest = tk.encode_batch_packed(texts, L, eos_id=src['eos'], **ALL)
            assert device_summary(batch, rest, L) == strip(src['one'][bi][str(L)]), (bi, L)
            carry = None
            for part, rec in zip((texts[:c1], texts[c1:c2], texts[c2:]), src['chain'][bi][str(L)]):
                batch, carry = tk.encode_batch_packed(part, L, eos_id=src['eos'], carry=carry, **ALL)
                assert device_summary(batch, carry, L) == strip(rec), (bi, L)


def np_pack(S, starts, L, sep=-100):
    """the oracle, vectorised: S int64 stream, starts the document starts -> (input_ids, labels, position_ids, seq_idx,
    cu_seq_lens, max_length, rest ids, rest splits), flat"""
    T = S.size
    NL = T // L * L
    first = np.zeros(NL, bool)
    first[::L] = True
    first[starts[starts < NL]] = True
    ps = np.flatnonzero(first)
    seq = np.cumsum(first) - 1
    pos = np.arange(NL) - ps[seq]
    labels = np.where(pos == 0, sep, S[:NL])
    cu = np.append(ps, NL)
    rsp = np.concatenate([[0], starts[(starts > NL) & (starts < T)] - NL, [T - NL]]) if T > NL else np.zeros(1, np.int64)
    return S[:NL], labels, pos, seq.astype(np.int32), cu.astype(np.int32), int(np.diff(cu).max()) if NL else 0, S[NL:], rsp


def np_stream(values, splits, eos):
    """the stream of (values, splits) rows with eos after every row, and its document starts"""
    v = values.astype(np.int64)
    lens = np.diff(splits)
    if eos is None:
        S = v[splits[0]:splits[-1]]
        starts = (splits[:-1] - splits[0])[lens > 0]
    else:
        S = np.insert(v[splits[0]:splits[-1]], splits[1:] - splits[0], eos)
        starts = splits[:-1] - splits[0] + np.arange(lens.size)
    return S, starts


def check_against_np(batch, rest, want, L):
    ids, labels, pos, seq, cu, longest, rv, rs = want
    n = ids.size // L
    assert tuple(batch['input_ids'].shape) == (n, L)
    assert np.array_equal(batch['input_ids'].cpu().numpy().ravel(), ids)
    assert np.array_equal(batch['labels'].cpu().numpy().ravel(), labels)
    if 'position_ids' in batch:
        assert np.array_equal(batch['position_ids'].cpu().numpy().ravel(), pos)
    if 'seq_idx' in batch:
        assert np.array_equal(batch['seq_idx'].cpu().numpy().ravel(), seq)
    if 'cu_seq_lens_q' in batch:
        assert np.array_equal(batch['cu_seq_lens_q'].cpu().numpy(), cu) and batch['max_length_q'] == longest
    assert np.array_equal(rest.values.cpu().numpy(), rv) and np.array_equal(rest.splits.cpu().numpy(), rs)


@pytest.mark.gpu
def test_uint16_equals_int32_with_high_ids(A, toks):
    """compact ids (uint16 bit patterns in an int16 tensor, and a real uint16 tensor) against int32, ids >= 2^15 included"""
    import torch
    eng = toks['bpe24k']._eng
    rng = np.random.default_rng(7)
    lens = rng.integers(0, 40, 3000)
    lens[::17] = 0
    values = rng.integers(0, 65536, int(lens.sum()))
    splits = np.concatenate([[0], np.cumsum(lens)])
    for L, eos in ((1, None), (5, 65535), (64, 3), (4096, None)):
        want = np_pack(*np_stream(values, splits, eos), L)
        sp = torch.from_numpy(splits).to(eng.device)
        i32 = torch.from_numpy(values.astype(np.int32)).to(eng.device)
        c16 = torch.from_numpy(values.astype(np.uint16).view(np.int16)).to(eng.device)
        outs = [eng.pack_batch((t, sp), L, eos_id=eos, **ALL) for t in (i32, c16, c16.view(torch.uint16))]
        for batch, rest in outs:
            check_against_np(batch, rest, want, L)


@pytest.mark.gpu
def test_edge_batches(A, toks):
    import torch
    eng = toks['bpe24k']._eng
    dev = eng.device

    def rag(rows):
        return ragged_of(torch, rows, 'int32', dev)

    def check(rows, L, eos=None, carry=None, **kw):
        batch, rest = eng.pack_batch(rag(rows), L, eos_id=eos, carry=carry, **kw)
        cr = None if carry is None else ([int(x) for x in carry.values.cpu()], [int(x) for x in carry.splits.cpu()])
        pieces, want_rest = O.pack(rows, L, eos, cr)
        flat = O.flatten(pieces, kw.get('separator_id', -100))
        assert batch['input_ids'].view(-1).tolist() == flat['input_ids']
        assert batch['labels'].view(-1).tolist() == flat['labels']
        if kw.get('return_position_ids', True):
            assert batch['position_ids'].view(-1).tolist() == flat['position_ids']
        else:
            assert 'position_ids' not in batch
        if kw.get('return_seq_idx'):
            assert batch['seq_idx'].view(-1).tolist() == flat['seq_idx']
        else:
            assert 'seq_idx' not in batch
        if kw.get('return_flash_attn_kwargs'):
            assert batch['cu_seq_lens_q'].tolist() == flat['cu_seq_lens'] and batch['max_length_q'] == flat['max_length']
        else:
            assert 'cu_seq_lens_q' not in batch and 'max_length_q' not in batch
        assert (rest.values.tolist(), rest.splits.tolist()) == (list(want_rest[0]), list(want_rest[1]))
        return batch, rest

    b, r = check([], 4, **ALL)                                           # no rows
    assert b['input_ids'].shape == (0, 4) and b['cu_seq_lens_q'].tolist() == [0] and r.splits.tolist() == [0]
    check([[], [], []], 4, **ALL)                                        # only empty rows
    b, r = check([[], [], []], 2, eos=9, **ALL)                          # ... with eos: three 1-id documents
    assert b['input_ids'].tolist() == [[9, 9]] and r.values.tolist() == [9]
    b, r = check([[1, 2], [3]], 8, **ALL)                                # T < L: everything is rest
    assert b['input_ids'].shape == (0, 8) and r.splits.tolist() == [0, 2, 3]
    b, r = check([[1, 2], [3, 4, 5, 6]], 3, **ALL)                       # T a multiple of L: empty rest
    assert r.values.numel() == 0 and r.splits.tolist() == [0]
    b, _ = check([[1, 2, 3], [4], [5, 6]], 1, eos=0, **ALL)              # L = 1: every label is the separator
    assert set(b['labels'].view(-1).tolist()) == {-100}
    b, r = check([[7, 8, 9]], 2, carry=A.Ragged(torch.tensor([1, 2, 3], dtype=torch.int32, device=dev),
                                                 torch.tensor([0, 1, 3], dtype=torch.int64, device=dev)), **ALL)
    check([[1, 2, 3, 4, 5]], 2, separator_id=-1, **ALL)
    for flags in range(8):                                               # every combination of the return flags
        kw = dict(return_position_ids=bool(flags & 1), return_seq_idx=bool(flags & 2), return_flash_attn_kwargs=bool(flags & 4))
        check([[1, 2, 3], [], [4, 5, 6, 7, 8], [9]], 3, eos=2, **kw)
    # many empty rows between two documents: more units than a tile's window holds
    check([[1, 2]] + [[]] * 5000 + [[3, 4, 5]] + [[6]] * 700, 7, **ALL)
    check([[1, 2]] + [[]] * 5000 + [[3, 4, 5]] + [[6]] * 700, 7, eos=0, **ALL)


@pytest.mark.gpu
def test_one_8mb_row(A, toks):
    import torch
    eng = toks['bpe24k']._eng
    rng = np.random.default_rng(8)
    lens = np.array([3, 8 << 20, 5])
    values = rng.integers(0, 24000, int(lens.sum()))
    splits = np.concatenate([[0], np.cumsum(lens)])
    batch, rest = eng.pack_batch((torch.from_numpy(values.astype(np.int32)).to(eng.device), torch.from_numpy(splits).to(eng.device)),
                                 128, **ALL)
    check_against_np(batch, rest, np_pack(*np_stream(values, splits, None), 128), 128)


@pytest.mark.gpu
def test_refusals_leave_the_engine_usable(A, toks):
    import torch
    eng = toks['bpe24k']._eng
    dev = eng.device
    ids = (torch.tensor([5, 6, 7], dtype=torch.int32, device=dev), torch.tensor([0, 1, 3], dtype=torch.int64, device=dev))
    for kw in (dict(block_size=0), dict(block_size=-3), dict(block_size=2.0), dict(block_size=2, eos_id=-1),
               dict(block_size=2, eos_id=2 ** 31), dict(block_size=2, carry=[1, 2]),
               dict(block_size=2, carry=(torch.zeros(1, dtype=torch.int64, device=dev), torch.zeros(2, dtype=torch.int64, device=dev))),
               dict(block_size=2, carry=(torch.zeros(1, dtype=torch.int32), torch.zeros(2, dtype=torch.int64))),
               dict(block_size=2, carry=(torch.zeros(1, dtype=torch.int32, device=dev), torch.zeros(0, dtype=torch.int64, device=dev))),
               dict(block_size=2, carry=(torch.zeros(1, dtype=torch.int32, device=dev),))):
        with pytest.raises(ValueError):
            eng.pack_batch(ids, **kw)
    # a stream of 2^31 ids: refused on the device from the splits (no ids behind them are read)
    big = torch.tensor([0, 2 ** 30, 2 ** 31 - 1], dtype=torch.int64, device=dev)
    with pytest.raises(ValueError, match='2\\^31'):
        eng.pack_batch((ids[0], big), 8, eos_id=2)
    batch, rest = eng.pack_batch(ids, 2, **ALL)
    assert batch['input_ids'].tolist() == [[5, 6]] and batch['labels'].tolist() == [[-100, -100]]
    assert rest.values.tolist() == [7] and rest.splits.tolist() == [0, 1]


@pytest.mark.gpu
@pytest.mark.parametrize('kind,model,eos', [('hinglish', 'bpe24k.json', None), ('hindi', 'spm24k.model', 2)])
def test_pack_at_64mb_equals_numpy_oracle(A, kind, model, eos):
    """64 MB of synthetic text, encoded, packed with L = 2048 and 8192 (and 3) in one call and in a 4-call chain, against
    the vectorised oracle"""
    import torch
    import synth_corpus as sc
    tk = A.aksharTokenizer(os.path.join(MODELS, model), 'bpe' if model.endswith('.json') else 'sentencepiece')
    eng = tk._eng
    data, off = sc.Corpus(kind, 64).generate(64 << 20)
    enc, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), tk.model.kind)
    values, splits = enc.values.cpu().numpy(), enc.splits.cpu().numpy()
    S, starts = np_stream(values, splits, eos)
    n = splits.size - 1
    for L in (3, 2048, 8192):
        want = np_pack(S, starts, L)
        batch, rest = eng.pack_batch(enc, L, eos_id=eos, **ALL)
        check_against_np(batch, rest, want, L)
        cuts = [0, n // 7, n // 2, n // 2 + 1, n]
        carry, got = None, []
        for lo, hi in zip(cuts, cuts[1:]):
            b, carry = eng.pack_batch((enc.values, enc.splits[lo:hi + 1]), L, eos_id=eos, carry=carry)
            got.append(b)
        for k in ('input_ids', 'labels', 'position_ids'):
            assert torch.equal(torch.cat([b[k] for b in got]), batch[k]), (L, k)
        assert torch.equal(carry.values, rest.values) and torch.equal(carry.splits, rest.splits)


@pytest.mark.gpu
def test_pack_lines_equals_one_call(A, tmp_path):
    """pack_lines over a 256 MiB file read in 4 or more pieces equals pack_batch over the whole file's ids in one call"""
    import torch
    import synth_corpus as sc
    from akshar_b200 import corpus
    tk = A.aksharTokenizer(os.path.join(MODELS, 'bpe24k.json'), 'bpe')
    data, off = sc.Corpus('hinglish', 256).generate(256 << 20)
    path = tmp_path / 'corpus.txt'
    np.insert(data, off[1:-1], np.uint8(10)).tofile(str(path))
    del data, off
    chunk = 48 << 20
    pieces = corpus.encode_lines(tk, str(path), as_device=True, chunk_bytes=chunk)
    assert len(pieces) >= 4
    values = torch.cat([p.values for p in pieces])
    lens = torch.cat([p.splits[1:] - p.splits[:-1] for p in pieces])
    splits = torch.cat([torch.zeros(1, dtype=torch.int64, device=values.device), torch.cumsum(lens, 0)])
    del pieces
    L = 2048
    whole, _ = tk._eng.pack_batch((values, splits), L, **ALL)
    got = list(corpus.pack_lines(tk, str(path), L, chunk_bytes=chunk, **ALL))
    assert len(got) >= 4
    for k in ('input_ids', 'labels', 'position_ids'):
        assert torch.equal(torch.cat([b[k] for b in got]), whole[k]), k
    seq = torch.cat([b['seq_idx'] + int(sum(b2['cu_seq_lens_q'].numel() - 1 for b2 in got[:i])) for i, b in enumerate(got)])
    assert torch.equal(seq, whole['seq_idx'])
    cu = torch.cat([got[0]['cu_seq_lens_q'][:1]] + [b['cu_seq_lens_q'][1:] + int(sum(b2['input_ids'].numel() for b2 in got[:i]))
                                                    for i, b in enumerate(got)])
    assert torch.equal(cu, whole['cu_seq_lens_q'])
    assert max(b['max_length_q'] for b in got) == whole['max_length_q']
