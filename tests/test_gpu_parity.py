"""Parity of the CUDA path (through the C ABI) with the reference -- run with `-m gpu` on a B200.

Bar: bit-exact records (integer/index work).  Sources of truth, in order:
  1. tests/golden/*.json  -- produced by the unmodified reference (both flavours);
  2. oracle.OracleAutomaton -- the pinned C restatement, on seeded random batches at sizes it
     finishes in seconds; the compiled reference too, as recorded in tests/golden/reference;
  3. at BASELINE.json's full sizes: properties that need no CPU run -- every planted
     occurrence is reported, no duplicates, each reported record really is an occurrence
     (sampled), and the two independent kernels (filter / DFA) agree exactly.
"""
import numpy as np
import pytest

import oracle
import pyahocorasick_b200 as ac
from golden_driver import all_scenarios, run_ops
from pyahocorasick_b200 import automaton as am
from pyahocorasick_b200 import synth
from recorded_reference import reference_records  # noqa: F401 -- fixture

pytestmark = pytest.mark.gpu
B = ac.flavour("bytes")

SC = all_scenarios()


@pytest.mark.parametrize("algo", ["filter", "dfa"])
@pytest.mark.parametrize("sc", SC, ids=[s["name"] for s in SC])
def test_golden_on_gpu(sc, algo, monkeypatch):
    real = am.Automaton._scan_flat

    def forced(self, flat, offsets, n_hay, stride_bytes, algo="auto", sort=True, device=None, narrow=False, _a=algo, **kw):
        return real(self, flat, offsets, n_hay, stride_bytes, algo=_a if algo == "auto" else algo, sort=sort, device=device, narrow=narrow, **kw)
    monkeypatch.setattr(am.Automaton, "_scan_flat", forced)
    bad = run_ops(ac.flavour(sc["flavour"]), sc, record=False)
    assert not bad, bad[:3]


def _oracle_for(keys):
    O = oracle.OracleAutomaton()
    for i, k in enumerate(keys):
        O.add_word(k, i)
    O.make_automaton()
    return O


def _records(m):
    return list(zip(m.hay_id.tolist(), m.end_index.tolist(), m.key_id.tolist()))


def _want_sorted(O, keys, flat, off):
    rec = O.scan_batch_bytes(flat, off).tolist()
    # oracle order inside one (hay, end) is fail-chain order = longest key first: already what sort=True gives
    return [tuple(r) for r in rec]


CASES = [
    # name, alphabet, n_keys, (lo, hi), n_hay, hay_len
    ("alnum_4_16", synth.ALNUM, 10_000, (4, 16), 4000, 256),
    ("alnum_1_5", synth.ALNUM, 300, (1, 5), 500, 300),
    ("ab_1_8", np.frombuffer(b"ab", dtype=np.uint8), 40, (1, 8), 300, 500),
    ("dna_20", synth.DNA, 5000, (20, 20), 3000, 150),
    ("dna_8_12", synth.DNA, 3000, (8, 12), 1000, 150),
    ("allbytes_2_6", np.arange(256, dtype=np.uint8), 5000, (2, 6), 1000, 777),
    ("hi_bytes", np.array([0, 1, 127, 128, 200, 255], dtype=np.uint8), 200, (1, 6), 500, 333),
    ("long_keys", synth.ALNUM, 2000, (17, 40), 800, 1000),
]


@pytest.mark.parametrize("algo", ["filter", "dfa"])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_random_batches_match_oracle(case, algo):
    name, alpha, nk, (lo, hi), nh, hl = case
    rng = np.random.Generator(np.random.PCG64(sum(name.encode()) * 7919))
    keys = synth.draw_keys(rng, alpha, nk, lo, hi)
    hay = synth.random_haystacks(rng, alpha, nh, hl)
    synth.plant(rng, hay, keys, np.arange(0, nh, 2))
    A = synth.build_automaton(keys)
    O = _oracle_for(keys)
    # fixed stride
    off = np.arange(nh + 1, dtype=np.int64) * hl
    want = _want_sorted(O, keys, hay.reshape(-1), off)
    assert len(want) > 0
    got = _records(A.find_all_batch(hay, algo=algo))
    assert got == want
    # ragged offsets, with empty haystacks and odd alignment
    cuts = np.sort(rng.integers(0, hay.size + 1, size=nh))
    cuts[5::7] = cuts[4::7][:len(cuts[5::7])]                 # repeated offsets = empty haystacks
    roff = np.concatenate([[0, 0], np.sort(cuts), [hay.size, hay.size]]).astype(np.int64)
    want2 = _want_sorted(O, keys, hay.reshape(-1), roff)
    got2 = _records(A.find_all_batch((hay.reshape(-1), roff), algo=algo))
    assert got2 == want2
    # list-of-bytes entry point
    hs = [hay[i, : int(rng.integers(0, hl + 1))].tobytes() for i in range(0, min(nh, 200))]
    loff = np.concatenate([[0], np.cumsum([len(h) for h in hs])]).astype(np.int64)
    lflat = np.frombuffer(b"".join(hs), dtype=np.uint8)
    want3 = _want_sorted(O, keys, lflat, loff) if lflat.size else []
    assert _records(A.find_all_batch(hs, algo=algo)) == want3


def _reference_batch(keys, rows):
    def compute(ref):
        R = ref.Automaton(ref.STORE_INTS)
        for i, k in enumerate(keys):
            R.add_word(k, i)
        R.make_automaton()
        return oracle.ref_scan_batch(R, [row.tobytes() for row in rows])
    return compute


def test_reference_extension_agrees_on_c2_sample(reference_records):
    """The unmodified reference on a C2 sub-sample."""
    w = synth.make("C2", scale=0.005)
    A = synth.build_automaton(w.keys)
    want = reference_records("c2_sample", _reference_batch(w.keys, w.haystacks))
    for algo in ("filter", "dfa"):
        m = A.find_all_batch(w.haystacks, algo=algo)
        assert list(zip(m.hay_id.tolist(), m.end_index.tolist(), m.values())) == want


def test_iter_long_batch_matches_oracle():
    """find_long_batch == looping the oracle's iter_long (pinned to the reference by tests/golden) per haystack."""
    rng = np.random.Generator(np.random.PCG64(2024))
    for alpha, nk, lo, hi in ((np.frombuffer(b"ab", dtype=np.uint8), 30, 1, 6), (synth.ALNUM, 3000, 2, 8), (synth.DNA, 500, 3, 10)):
        keys = synth.draw_keys(rng, alpha, nk, lo, hi)
        hay = synth.random_haystacks(rng, alpha, 400, 200)
        synth.plant(rng, hay, keys, np.arange(400))
        A = synth.build_automaton(keys)
        O = _oracle_for(keys)
        want = [(h, e, v) for h in range(400) for e, v in O.iter_long(hay[h].tobytes())]
        m = A.find_long_batch(hay)
        assert list(zip(m.hay_id.tolist(), m.end_index.tolist(), m.values())) == want
        assert list(A.iter_long(hay[7].tobytes(), 3, 150)) == O.iter_long(hay[7].tobytes(), 3, 150)


def test_pathological_overlaps():
    keys = [b"a" * k for k in range(1, 33)] + [b"a" * 31 + b"b", b"ba", b"ab"]
    A = synth.build_automaton(keys)
    O = _oracle_for(keys)
    hay = np.frombuffer((b"a" * 200 + b"b") * 20, dtype=np.uint8).reshape(1, -1).copy()
    off = np.array([0, hay.size], dtype=np.int64)
    want = _want_sorted(O, keys, hay.reshape(-1), off)
    for algo in ("filter", "dfa"):
        assert _records(A.find_all_batch(hay, algo=algo)) == want


def test_pair_kernel_boundaries_and_dense_text():
    """the PAIR kernel (gram 4, stride 1): occurrences across every kind of boundary it has -- the 16-byte runs of a
    lane, the two halves of a 1 KiB slice, slices, tiles -- and text dense enough to overflow its item list (more than
    64 pending positions in a slice) and its candidate ring (more than 64 candidates in a slice), against the oracle"""
    rng = np.random.Generator(np.random.PCG64(20260923))
    keys = synth.draw_keys(rng, synth.ALNUM, 600, 4, 16)
    A = synth.build_automaton(keys)
    f = A.flat()
    assert f["filter_flags"] & 2 and f["gram_bytes"] == 4 and f["stride"] == 1          # PAIR placement -> acb_pair_kernel
    O = _oracle_for(keys)
    n = 200 * 1024 + 37                                                                # ten 20 KiB tiles and a ragged tail
    hay = rng.choice(np.frombuffer(b"#%&*+-", dtype=np.uint8), size=n).astype(np.uint8)    # no key letter: only planted keys match
    k = 0
    for b in range(16, n - 32, 16):                                                     # every run / half / slice / tile boundary ...
        key = np.frombuffer(keys[k % len(keys)], dtype=np.uint8)
        start = b - 1 - (k % min(15, len(key) - 1))                                     # ... is crossed by a key
        if (b // 16) % 3 == 0:
            hay[start:start + len(key)] = key
        k += 1
    hay[n - 4:] = np.frombuffer(keys[[len(x) for x in keys].index(4)], dtype=np.uint8)  # a key that ends with the buffer
    off = np.array([0, n], dtype=np.int64)
    want = _want_sorted(O, keys, hay, off)
    assert len(want) > 3000
    assert _records(A.find_all_batch((hay, off), algo="filter")) == want
    roff = np.concatenate([[0], np.sort(rng.integers(0, n, size=300)), [n]]).astype(np.int64)
    assert _records(A.find_all_batch((hay, roff), algo="filter")) == _want_sorted(O, keys, hay, roff)
    # dense text: one short key back to back -- every position of a slice is pending, every one is a candidate
    dense_keys = [b"abab", b"baba", b"ababab", b"abcd"]
    D = synth.build_automaton(dense_keys)
    assert D.flat()["filter_flags"] & 2
    OD = _oracle_for(dense_keys)
    dh = np.frombuffer(b"ab" * 30000 + b"abcd" * 100 + b"ab" * 5000, dtype=np.uint8).copy()
    doff = np.array([0, 1000, 1001, 40000, dh.size], dtype=np.int64)
    assert _records(D.find_all_batch((dh, doff), algo="filter")) == _want_sorted(OD, dense_keys, dh, doff)


def test_unicode_and_sequence_flavours_on_gpu():
    U = ac.flavour("unicode")
    A = U.Automaton()
    words = ["wy", "ważyć", "aż", "waży", "ż", "中文", "\U0001F629", "a\U0001F629b"]
    for i, w in enumerate(words):
        A.add_word(w, (i, w))
    A.make_automaton()
    text = "wyważyć 中文 a\U0001F629b ż" * 50
    Ro = oracle.OracleAutomaton()
    for i, w in enumerate(words):
        Ro.add_word(w, i)
    Ro.make_automaton()
    want = [(e, (v, words[v])) for e, v in Ro.find_all(text)]
    assert list(A.iter(text)) == want
    S = U.Automaton(U.STORE_INTS, U.KEY_SEQUENCE)
    seqs = [(1, 2, 3), (2, 3), (2 ** 32 - 1, 0), (70000, 1)]
    for i, s in enumerate(seqs):
        S.add_word(s, i)
    S.make_automaton()
    hay = (0, 1, 2, 3, 2 ** 32 - 1, 0, 70000, 1, 2, 3) * 30
    So = oracle.OracleAutomaton()
    for i, s in enumerate(seqs):
        So.add_word(s, i)
    So.make_automaton()
    assert list(S.iter(hay)) == So.find_all(hay)


# ------------------------------------------------------------------ BASELINE.json sizes
def _check_full(w, A, sample=20000):
    m_f = A.find_all_batch(w.haystacks, algo="filter")
    rec_f = np.stack([m_f.hay_id, m_f.end_index, m_f.key_id], axis=1).astype(np.int64)
    # (1) every planted occurrence is reported
    stride = w.haystacks.shape[1]
    def pack(h, e, k):
        return (h * stride + e) * (len(w.keys) + 1) + k
    got = pack(rec_f[:, 0], rec_f[:, 1], rec_f[:, 2])
    planted = pack(w.planted_hay, w.planted_end, w.planted_key)
    assert np.isin(planted, got).all()
    # (2) no duplicates
    assert len(np.unique(got)) == len(got)
    # (3) sortedness in the reference's order
    klen = np.fromiter((len(k) for k in w.keys), dtype=np.int64, count=len(w.keys))
    order = np.lexsort((-klen[rec_f[:, 2]], rec_f[:, 1], rec_f[:, 0]))
    assert (order == np.arange(len(order))).all()
    # (4) a sample of reported records really are occurrences
    rng = np.random.Generator(np.random.PCG64(7))
    for i in rng.integers(0, len(rec_f), size=min(sample, len(rec_f))).tolist():
        h, e, k = rec_f[i]
        key = w.keys[k]
        assert w.haystacks[h, e - len(key) + 1:e + 1].tobytes() == key
    # (5) the independent DFA kernel agrees exactly
    m_d = A.find_all_batch(w.haystacks, algo="dfa")
    assert np.array_equal(m_d.hay_id, m_f.hay_id) and np.array_equal(m_d.end_index, m_f.end_index) and np.array_equal(m_d.key_id, m_f.key_id)
    return len(got)


def _check_reference_rows(w, A, rows, reference_records):
    """the compiled reference over the listed haystacks: identical records in identical order"""
    sub = np.ascontiguousarray(w.haystacks[rows])
    want = reference_records("rows", _reference_batch(w.keys, sub))
    m = A.find_all_batch(sub)
    assert list(zip(m.hay_id.tolist(), m.end_index.tolist(), m.values())) == want


def test_full_size_c2_properties(reference_records):
    w = synth.make("C2", scale=1.0)
    A = synth.build_automaton(w.keys)
    n = _check_full(w, A)
    assert n >= w.n_hay
    _check_reference_rows(w, A, np.arange(0, w.n_hay, 10), reference_records)   # every 10th haystack: 100 k, BASELINE.md section 2


def test_full_size_c3_dna_properties(reference_records):
    w = synth.make("C3", scale=1.0)          # BASELINE config 3 at its stated size: 10 M reads x 150 B, 100 k 20-mers
    A = synth.build_automaton(w.keys)
    _check_full(w, A)
    _check_reference_rows(w, A, np.arange(0, w.n_hay, 100), reference_records)  # 100 k reads through the reference


def test_full_size_c4_long_haystacks_properties(reference_records):
    w = synth.make("C4", scale=1.0)          # BASELINE config 4 at its stated size: 64 x 16 MiB, a key across every 16 KiB
    A = synth.build_automaton(w.keys)
    # more straddlers, one across every boundary the kernel or the host pipeline has: 512-byte slices of a tile, the
    # tiles themselves, and the 32 MiB chunks of the pipelined host scan (minus the reach of the longest key)
    flat = w.haystacks.reshape(-1)
    rng = np.random.Generator(np.random.PCG64(44))
    size = w.haystacks.shape[1]
    extra_h, extra_e, extra_k = [], [], []
    cuts = list(range(31 * 1024, flat.size, 31 * 1024 * 37)) + [c * (32 << 20) - d for c in range(1, flat.size >> 25) for d in (0, 32)]
    for b in cuts:
        if b <= 64 or b >= flat.size - 64 or b % size < 32 or b % size > size - 32:
            continue
        kid = int(rng.integers(0, len(w.keys)))
        k = np.frombuffer(w.keys[kid], dtype=np.uint8)
        st = b - int(rng.integers(1, len(k)))
        flat[st:st + len(k)] = k
        extra_h.append(st // size); extra_e.append(st % size + len(k) - 1); extra_k.append(kid)
    klen = np.fromiter((len(k) for k in w.keys), dtype=np.int64, count=len(w.keys))
    ph = np.concatenate([w.planted_hay, np.asarray(extra_h, dtype=np.int64)])
    pe = np.concatenate([w.planted_end, np.asarray(extra_e, dtype=np.int64)])
    pk = np.concatenate([w.planted_key, np.asarray(extra_k, dtype=np.int64)])
    starts = ph * size + pe - klen[pk] + 1                              # keep only plants whose bytes survived the new ones
    ok = np.ones(len(ph), dtype=bool)
    for L in np.unique(klen[pk]).tolist():
        sel = np.nonzero(klen[pk] == L)[0]
        got = flat[starts[sel][:, None] + np.arange(L)[None, :]]
        want = np.stack([np.frombuffer(w.keys[int(k)], dtype=np.uint8) for k in pk[sel]])
        ok[sel] = (got == want).all(axis=1)
    w.planted_hay, w.planted_end, w.planted_key = ph[ok], pe[ok], pk[ok]
    assert len(extra_h) > 40
    _check_full(w, A)
    _check_reference_rows(w, A, np.array([1]), reference_records)     # one whole 16 MiB haystack through the reference


def test_c5_100k_keys_properties(reference_records):
    w = synth.make("C5", scale=0.125)        # 1 M x 256 B (one GPU's shard of BASELINE config 5), 100 k keys
    A = synth.build_automaton(w.keys)
    _check_full(w, A)
    _check_reference_rows(w, A, np.arange(0, w.n_hay, 10), reference_records)


def test_dense_matches_grow_the_buffers():
    """a key set that matches at every position: the match buffer overflows and is regrown, the internal
    candidate list falls back to its worst-case size; results still equal the oracle's."""
    keys = [b"a", b"aa", b"ab"]
    A = synth.build_automaton(keys)
    O = _oracle_for(keys)
    hay = np.full((64, 4096), ord("a"), dtype=np.uint8)
    hay[:, ::97] = ord("b")
    off = np.arange(65, dtype=np.int64) * 4096
    want = _want_sorted(O, keys, hay.reshape(-1), off)
    assert len(want) > 2 * hay.size * 0.9
    for algo in ("filter", "dfa"):
        assert _records(A.find_all_batch(hay, algo=algo)) == want
    import torch
    assert _records(A.find_all_batch(torch.from_numpy(hay).cuda())) == want       # device-resident entry, same growth path


def test_torch_cuda_tensor_batches():
    import torch
    w = synth.make("C2", scale=0.01)
    A = synth.build_automaton(w.keys)
    want = _records(A.find_all_batch(w.haystacks))
    d = torch.from_numpy(w.haystacks).cuda()
    for algo in ("filter", "dfa"):
        assert _records(A.find_all_batch(d, algo=algo)) == want
    assert sorted(_records(A.find_all_batch(d, sort=False))) == sorted(want)


def test_batch_larger_than_one_segment():
    """> 2 GiB in one call: the filter path scans it in 2 GiB segments (32-bit candidate offsets); a key planted
    across the segment boundary (inside one haystack) must be found, and both kernels must agree."""
    rng = np.random.Generator(np.random.PCG64(31))
    keys = synth.draw_keys(rng, synth.ALNUM, 2000, 4, 16)
    stride, n = 250, 9_000_000                                   # 2.25e9 bytes > 2^31
    hay = synth.random_haystacks(rng, synth.ALNUM, n, stride)
    rows = np.arange(0, n, 7)
    ph, pe, pk = synth.plant(rng, hay, keys, rows)
    flat = hay.reshape(-1)
    b = 1 << 31                                                  # straddle the segment boundary
    k = np.frombuffer(keys[5], dtype=np.uint8)
    st = b - len(k) // 2
    assert st // stride == (st + len(k) - 1) // stride           # stays inside one haystack
    flat[st:st + len(k)] = k
    w = synth.Workload("seg", keys, hay, np.append(ph, st // stride), np.append(pe, st % stride + len(k) - 1), np.append(pk, 5))
    # earlier plants in that haystack may have been overwritten: keep only plants whose bytes survived
    klen = np.fromiter((len(x) for x in keys), dtype=np.int64, count=len(keys))
    starts = w.planted_hay * stride + w.planted_end - klen[w.planted_key] + 1
    ok = np.ones(len(starts), dtype=bool)
    hit = np.nonzero(w.planted_hay == st // stride)[0]
    for i in hit.tolist():
        kk = np.frombuffer(keys[int(w.planted_key[i])], dtype=np.uint8)
        ok[i] = np.array_equal(flat[starts[i]:starts[i] + len(kk)], kk)
    w.planted_hay, w.planted_end, w.planted_key = w.planted_hay[ok], w.planted_end[ok], w.planted_key[ok]
    A = synth.build_automaton(keys)
    _check_full(w, A, sample=5000)


def test_device_resident_entry_and_overflow_retry():
    import ctypes
    import torch
    from pyahocorasick_b200 import _native as N
    w = synth.make("C2", scale=0.01)
    A = synth.build_automaton(w.keys)
    want = _records(A.find_all_batch(w.haystacks))
    tb = A._ensure_table(0)
    d_hay = torch.from_numpy(w.haystacks).cuda()
    d_cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    d_out = torch.empty((8, 3), dtype=torch.int32, device="cuda")            # far too small
    st = torch.cuda.current_stream().cuda_stream
    L = N.lib()
    N.check(L.acb_scan_device(tb, d_hay.data_ptr(), d_hay.numel(), None, w.n_hay, 256, d_out.data_ptr(), 8, d_cnt.data_ptr(), st, 0))
    torch.cuda.synchronize()
    assert int(d_cnt.item()) == len(want)                                    # counted, not stored
    d_out = torch.empty((len(want), 3), dtype=torch.int32, device="cuda")
    d_cnt.zero_()
    N.check(L.acb_scan_device(tb, d_hay.data_ptr(), d_hay.numel(), None, w.n_hay, 256, d_out.data_ptr(), len(want), d_cnt.data_ptr(), st, 0))
    torch.cuda.synchronize()
    got = sorted(map(tuple, d_out.cpu().numpy().tolist()))
    assert got == sorted(want)


@pytest.mark.gpu
def test_records_are_handed_over_without_a_copy_and_stay_valid():
    """acb_take_records: a result keeps its pinned buffer while any view of it is alive (a later scan must not
    overwrite it), and the buffer is reused once the result is dropped"""
    import gc
    w = synth.make("C2", scale=0.004)
    A = synth.build_automaton(w.keys)
    first = A.find_all_batch(w.haystacks)
    snap = (first.hay_id.copy(), first.end_index.copy(), first.key_id.copy())
    addr = first.end_index.__array_interface__["data"][0]
    other = A.find_all_batch(w.haystacks[::-1].copy())          # a different scan while `first` is still held
    assert other.end_index.__array_interface__["data"][0] != addr
    for got, want in zip((first.hay_id, first.end_index, first.key_id), snap):
        assert np.array_equal(got, want)
    again = A.find_all_batch(w.haystacks)
    for got, want in zip((again.hay_id, again.end_index, again.key_id), snap):
        assert np.array_equal(got, want)
    del first, other, again
    gc.collect()
    for _ in range(3):                                          # steady state: results dropped before the next call
        m = A.find_all_batch(w.haystacks)
        assert np.array_equal(m.end_index, snap[1])
        del m
        gc.collect()
