"""The reference's pickle tuple and `save` file format, both directions (SURVEY.md section 8(f) #2).

* golden: tests/golden/golden_serialized.json holds what the UNMODIFIED reference wrote
  (tests/golden/make_serialized.py); the drop-in must read it and answer like the reference did.
* differential (the reference as recorded in tests/golden/reference): what the drop-in writes, the reference must
  read; random key sets.
* malformed input is refused with the reference's exception types, never a crash.
"""
import base64
import json
import os
import pickle
import struct

import numpy as np
import pytest

import pyahocorasick_b200 as pkg
from pyahocorasick_b200 import serialize
from recorded_reference import reference  # noqa: F401 -- fixture

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "golden_serialized.json")))
STORES = {"STORE_ANY": 30, "STORE_INTS": 20, "STORE_LENGTH": 10}


def _conv(fl, s):
    return s.encode("latin-1") if fl == "bytes" else s


def _jvals(A):
    return sorted(json.dumps(v) for v in A.values())


def _check_against_scenario(A, sc):
    fl = sc["flavour"]
    assert A.kind == sc["kind"] and len(A) == sc["count"] and A.store == STORES[sc["store"]]
    assert _jvals(A) == sc["values_sorted"]
    if fl == "unicode":
        assert sorted([k, json.dumps(v)] for k, v in A.items()) == sc["items"]
    else:                                     # the drop-in's keys() do work in the bytes flavour
        want = [w.encode("latin-1") for w in GOLD["words"]]
        if sc["removed"]:
            want = [w for w in want if w not in (b"hers", b"abc")]
        assert sorted(A.keys()) == sorted(want)
    for w in GOLD["words"]:
        k = _conv(fl, w)
        gone = sc["removed"] and w in ("hers", "abc")
        assert A.exists(k) == (not gone)


@pytest.mark.parametrize("idx", range(len(GOLD["scenarios"])))
def test_reads_what_the_reference_wrote(idx, tmp_path, monkeypatch):
    sc = GOLD["scenarios"][idx]
    mod = pkg.flavour(sc["flavour"])
    chunks = [base64.b64decode(c) for c in sc["reduce_chunks"]]
    A = mod.Automaton(chunks, *sc["reduce_tail"], sc["reduce_values"])       # the 7-tuple constructor, src/Automaton.c:106-147
    _check_against_scenario(A, sc)
    p = tmp_path / "ref.save"
    p.write_bytes(base64.b64decode(sc["save_file"]))
    B = mod.load(str(p), pickle.loads)
    _check_against_scenario(B, sc)
    if sc["built"]:                            # search results: through the emulated device on CPU
        import emul
        emul.install(monkeypatch, "filter")
        hay = _conv(sc["flavour"], GOLD["hay"])
        for X in (A, B):
            assert [[e, json.dumps(v)] for e, v in X.iter(hay)] == sc["iter"]


def _build_pair(ref, fl, store, words, rng):
    mod = pkg.flavour(fl)
    A, R = mod.Automaton(store), ref.Automaton(store)
    for i, w in enumerate(words):
        if store == 30:
            v = {"i": i, "w": repr(w)}
            A.add_word(w, v), R.add_word(w, v)
        elif store == 20:
            v = int(rng.integers(-2 ** 31, 2 ** 31))
            A.add_word(w, v), R.add_word(w, v)
        else:
            A.add_word(w), R.add_word(w)
    return mod, ref, A, R


def _random_words(fl, rng, n):
    if fl == "bytes":
        al = np.frombuffer(b"abc\x80\xfe\xff", dtype=np.uint8)
        return list(dict.fromkeys(bytes(al[rng.integers(0, len(al), size=int(rng.integers(1, 7)))].tolist()) for _ in range(n)))
    al = "ab\xe9\u0142\U0001f600\uffff"
    return list(dict.fromkeys("".join(al[int(j)] for j in rng.integers(0, len(al), size=int(rng.integers(1, 7)))) for _ in range(n)))


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
@pytest.mark.parametrize("store", [30, 20, 10])
def test_the_reference_reads_what_we_write(fl, store, tmp_path, reference):
    rng = np.random.default_rng(1234 + store)
    for rnd in range(4):
        words = _random_words(fl, rng, 40)
        mod, ref, A, R = _build_pair(reference(fl), fl, store, words, rng)
        if rnd & 1:
            for w in words[::5]:
                assert A.remove_word(w) and R.remove_word(w)
        if rnd & 2:
            A.make_automaton(), R.make_automaton()
        hay = words[0] * 2 + b"".join(words[1:9]) if fl == "bytes" else words[0] * 2 + "".join(words[1:9])
        want_vals = sorted(map(repr, R.values()))
        # pickle tuple: ours -> reference, reference -> ours
        R2 = ref.Automaton(*serialize.reduce_args(A))
        A2 = mod.Automaton(*R.__reduce__()[1])
        assert R2.kind == A2.kind == R.kind and len(R2) == len(A2) == len(R)
        assert sorted(map(repr, R2.values())) == sorted(map(repr, A2.values())) == want_vals
        if fl == "unicode":
            assert sorted(R2.keys()) == sorted(A2.keys()) == sorted(R.keys())
        else:
            assert sorted(A2.keys()) == sorted(A.keys())
        for w in words:
            assert R2.exists(w) == A2.exists(w) == R.exists(w)
            if R.exists(w):
                assert repr(R2.get(w)) == repr(A2.get(w)) == repr(R.get(w))
        if R.kind == ref.AHOCORASICK:
            assert list(map(repr, R2.iter(hay))) == list(map(repr, R.iter(hay)))      # our fail links, followed by the reference
        # save files: ours -> reference, reference -> ours
        p1, p2 = str(tmp_path / f"a{rnd}"), str(tmp_path / f"b{rnd}")
        if store == 30:
            A.save(p1, pickle.dumps), R.save(p2, pickle.dumps)
        else:
            A.save(p1), R.save(p2)
        R3, A3 = ref.load(p1, pickle.loads), mod.load(p2, pickle.loads)
        assert R3.kind == A3.kind == R.kind and R3.store == A3.store == store
        assert sorted(map(repr, R3.values())) == sorted(map(repr, A3.values())) == want_vals
        if R.kind == ref.AHOCORASICK:
            assert list(map(repr, R3.iter(hay))) == list(map(repr, R.iter(hay)))
        # and plain pickle of the drop-in, either flavour
        P = pickle.loads(pickle.dumps(A))
        assert type(P) is type(A) and P.kind == A.kind and sorted(map(repr, P.values())) == want_vals


def test_key_sequence_and_empty_round_trips(tmp_path):
    for fl in ("bytes", "unicode"):
        mod = pkg.flavour(fl)
        A = mod.Automaton(mod.STORE_INTS, mod.KEY_SEQUENCE)
        keys = [(1, 2, 3), (1, 2), (65535, 7), (300, 300, 300, 9)]
        for i, k in enumerate(keys):
            A.add_word(k, i + 10)
        A.make_automaton()
        B = mod.Automaton(*serialize.reduce_args(A))
        assert B.kind == mod.AHOCORASICK and sorted(B.items()) == sorted(zip(keys, range(10, 14)))
        p = str(tmp_path / f"seq_{fl}")
        A.save(p)
        C = mod.load(p, pickle.loads)
        assert sorted(C.items()) == sorted(B.items()) and C.kind == mod.AHOCORASICK
        E = mod.Automaton()
        assert serialize.reduce_args(E) == () and pickle.loads(pickle.dumps(E)).kind == mod.EMPTY
        pe = str(tmp_path / f"empty_{fl}")
        E.save(pe, pickle.dumps)
        assert os.path.getsize(pe) == serialize.HEADER.size + serialize.FOOTER.size
        assert mod.load(pe, pickle.loads).kind == mod.EMPTY


def test_large_automaton_is_split_into_16MB_arrays_like_the_reference(reference):
    mod = pkg.flavour("bytes")
    rng = np.random.default_rng(5)
    A = mod.Automaton(mod.STORE_LENGTH)
    raw = rng.integers(97, 123, size=(60000, 12), dtype=np.uint8)
    for row in raw:
        A.add_word(row.tobytes())
    args = serialize.reduce_args(A)
    chunks = args[0]
    assert len(chunks) >= 2 and all(len(c) == serialize.CHUNK_BYTES for c in chunks[:-1]) and len(chunks[-1]) <= serialize.CHUNK_BYTES
    assert sum(struct.unpack_from("<q", c)[0] for c in chunks) == A.get_stats()["nodes_count"]
    B = mod.Automaton(*args)
    assert len(B) == len(A) and B.get_stats()["nodes_count"] == A.get_stats()["nodes_count"]
    assert all(B.get(row.tobytes()) == 12 for row in raw[::997])
    R = reference("bytes").Automaton(*args)
    assert len(R) == len(A) and all(R.get(row.tobytes()) == 12 for row in raw[::997])


def test_argument_rules_and_malformed_input(tmp_path):
    mod = pkg.flavour("bytes")
    A = mod.Automaton(mod.STORE_ANY)
    A.add_word(b"he", 1), A.add_word(b"she", 2)
    I = mod.Automaton(mod.STORE_INTS)
    I.add_word(b"he", 1)
    p = str(tmp_path / "x")
    # src/custompickle/pyhelpers.c:4-59
    with pytest.raises(ValueError, match="exactly two"):
        A.save(p)
    with pytest.raises(ValueError, match="exactly one"):
        I.save(p, pickle.dumps)
    with pytest.raises(TypeError, match="must be a string"):
        I.save(b"bytes-path")
    with pytest.raises(TypeError, match="callable"):
        A.save(p, 42)
    with pytest.raises(ValueError, match="exactly two"):
        mod.load(p)
    with pytest.raises(TypeError, match="serializer must return bytes"):
        A.save(p, lambda v: "text")
    with pytest.raises(OSError):
        mod.load(str(tmp_path / "missing"), pickle.loads)
    A.save(p, pickle.dumps)
    good = open(p, "rb").read()
    for bad, exc in ((b"X" + good[1:], ValueError), (good[:-1] + b"X", ValueError), (good[:60] + good[-24:], ValueError),
                     (good[:20], OSError)):
        open(p, "wb").write(bad)
        with pytest.raises(exc):
            mod.load(p, pickle.loads)
    huge = good[:-24] + struct.pack("<Q", 1 << 50) + good[-16:]     # footer announces 2^50 nodes
    open(p, "wb").write(huge)
    with pytest.raises(ValueError, match="nodes announced"):
        mod.load(p, pickle.loads)
    # constructor (src/Automaton.c:106-147, src/Automaton_pickle.c:270-303)
    args = serialize.reduce_args(A)
    with pytest.raises(TypeError, match="Expected list"):
        mod.Automaton(tuple(args[0]), *args[1:])
    with pytest.raises(ValueError):
        mod.Automaton(args[0], 7, *args[2:])                       # kind
    with pytest.raises(ValueError):
        mod.Automaton(args[0], args[1], 31, *args[3:])             # store
    with pytest.raises(ValueError, match="not a bytes object"):
        mod.Automaton(["text"], *args[1:])
    with pytest.raises(ValueError, match="not positive"):
        mod.Automaton([struct.pack("<q", 0) + args[0][0][8:]], *args[1:])
    with pytest.raises(ValueError):
        mod.Automaton([args[0][0][:-5]], *args[1:])                # truncated
    broken = bytearray(args[0][0])
    broken[8 + 24 + 2:8 + 24 + 10] = struct.pack("<Q", 999)        # first child of the root -> node 999
    with pytest.raises(ValueError):
        mod.Automaton([bytes(broken)], *args[1:])
    loop = bytearray(args[0][0])
    loop[8 + 24 + 2:8 + 24 + 10] = struct.pack("<Q", 1)            # ... -> the root itself
    with pytest.raises(ValueError):
        mod.Automaton([bytes(loop)], *args[1:])
    with pytest.raises(IndexError):
        mod.Automaton(args[0], *args[1:6], [])                     # values list too short


# ------------------------------------------------------------------ the flat-table cache (SURVEY 8(f) #2, last clause)
def _flat_equal(a, b):
    return all(np.array_equal(a[k], b[k]) if isinstance(a[k], np.ndarray) else a[k] == b[k] for k in a)


def test_flat_table_cache_round_trip_and_rejections(tmp_path, monkeypatch):
    """a second load of the same file installs the cached tables instead of rebuilding them; a cache that belongs to
    another key set, another library version or is damaged is refused and the automaton is built the long way"""
    import ctypes
    from pyahocorasick_b200 import _native as N
    from pyahocorasick_b200 import synth
    mod = pkg.flavour("bytes")
    keys = synth.draw_keys(np.random.Generator(np.random.PCG64(9)), synth.ALNUM, 3000, 4, 12)
    A = mod.Automaton(mod.STORE_INTS)
    for i, k in enumerate(keys):
        A.add_word(k, i)
    A.make_automaton()
    path = str(tmp_path / "a.save")
    A.save(path)
    assert not os.path.exists(path + ".acb200")
    B = mod.load(path, pickle.loads)                                  # miss: builds, writes the cache
    assert os.path.exists(path + ".acb200")
    calls = []
    real = mod.Automaton.make_automaton
    monkeypatch.setattr(mod.Automaton, "make_automaton", lambda self: (calls.append(1), real(self))[1])
    C = mod.load(path, pickle.loads)                                  # hit: make_automaton is never called
    assert calls == [] and C.kind == pkg.AHOCORASICK
    assert _flat_equal(B.flat(), C.flat()) and sorted(C.items()) == sorted(B.items())
    # the same cache offered to a different key set: refused by the content hash, built the long way
    D = mod.Automaton(mod.STORE_INTS)
    for i, k in enumerate(keys[:-1]):
        D.add_word(k, i)
    D._make_automaton_cached(path + ".acb200")
    assert calls == [1] and D.kind == pkg.AHOCORASICK
    # damaged cache files: truncated, flipped magic -> rebuilt (and the cache rewritten)
    blob = open(path + ".acb200", "rb").read()
    for bad in (blob[:len(blob) // 2], b"X" + blob[1:], blob[:600]):
        open(path + ".acb200", "wb").write(bad)
        calls.clear()
        E = mod.load(path, pickle.loads)
        assert calls == [1] and _flat_equal(E.flat(), B.flat())
    # the C entry points by themselves
    L = N.lib()
    need = ctypes.c_int64(0)
    T = mod.Automaton(mod.STORE_INTS)
    T.add_word(b"abc", 0)
    assert L.acb_trie_flat_save(T._trie, None, 0, ctypes.byref(need)) == N.ACB_ESTATE     # not built yet
    assert L.acb_trie_content_hash(T._trie) != L.acb_trie_content_hash(B._trie)


def test_unpickling_uses_the_cache_directory(tmp_path, monkeypatch):
    mod = pkg.flavour("unicode")
    A = mod.Automaton()
    for w in GOLD["words"]:
        A.add_word(w, w.upper())
    A.make_automaton()
    blob = pickle.dumps(A)
    monkeypatch.setenv("ACB200_CACHE_DIR", str(tmp_path))
    B = pickle.loads(blob)
    assert len(list(tmp_path.glob("*.acb200"))) == 1
    calls = []
    real = mod.Automaton.make_automaton
    monkeypatch.setattr(mod.Automaton, "make_automaton", lambda self: (calls.append(1), real(self))[1])
    C = pickle.loads(blob)
    assert calls == [] and C.kind == pkg.AHOCORASICK and _flat_equal(B.flat(), C.flat())


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(len(GOLD["scenarios"])))
def test_loaded_automata_search_on_the_gpu(idx, tmp_path):
    """every automaton the reference serialised, read back (twice: the second load comes from the flat-table cache)
    and searched on the real kernels"""
    sc = GOLD["scenarios"][idx]
    if not sc["built"]:
        pytest.skip("not an automaton")
    mod = pkg.flavour(sc["flavour"])
    p = tmp_path / "ref.save"
    p.write_bytes(base64.b64decode(sc["save_file"]))
    hay = _conv(sc["flavour"], GOLD["hay"])
    for _ in range(2):
        B = mod.load(str(p), pickle.loads)
        assert [[e, json.dumps(v)] for e, v in B.iter(hay)] == sc["iter"]
    assert os.path.exists(str(p) + ".acb200")
