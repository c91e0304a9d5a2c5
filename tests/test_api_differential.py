"""Host-side API of the drop-in (everything that is not a search) compared call by call with the
unmodified reference extension, both flavours, as recorded in tests/golden/reference (tests/recorded_reference.py).
CPU only."""
import numpy as np
import pytest

import pyahocorasick_b200 as ac
from recorded_reference import reference  # noqa: F401 -- fixture


def _conv(fl, s):
    return s if fl == "unicode" else s.encode("utf-8")


def _call(obj, name, *args):
    try:
        r = getattr(obj, name)(*args)
        if name in ("keys", "values", "items"):
            r = list(r)            # NOT sorted: the order is the reference's trie walk (acb_trie_key_order)
        return ("ok", r)
    except Exception as e:  # noqa: BLE001
        return ("exc", type(e).__name__)


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_operation_sequences(fl, seed, reference):
    ref = reference(fl)
    mine = ac.flavour(fl)
    rng = np.random.Generator(np.random.PCG64(seed))
    R, M = ref.Automaton(), mine.Automaton()
    alphabet = "abé" if fl == "unicode" else "abc"
    pool = ["".join(alphabet[i] for i in rng.integers(0, 3, size=int(rng.integers(0, 5)))) for _ in range(40)]
    # the reference asserts (and exits) when trie_find / trie_longest run on an EMPTY automaton (root == NULL,
    # src/common.h:83-88): give both a first key so that the root exists for the whole sequence
    R.add_word(_conv(fl, "seed"), -1)
    M.add_word(_conv(fl, "seed"), -1)
    for step in range(400):
        w = _conv(fl, pool[int(rng.integers(0, len(pool)))])
        op = ["add_word", "remove_word", "pop", "exists", "match", "longest_prefix", "get", "get_default",
              "len", "kind", "make_automaton", "keys", "keys_prefix", "items", "contains"][int(rng.integers(0, 15))]
        if op == "add_word":
            a, b = _call(R, "add_word", w, step), _call(M, "add_word", w, step)
        elif op == "get_default":
            a, b = _call(R, "get", w, "dflt"), _call(M, "get", w, "dflt")
        elif op == "len":
            a, b = ("ok", len(R)), ("ok", len(M))
        elif op == "kind":
            a, b = ("ok", R.kind), ("ok", M.kind)
        elif op == "make_automaton":
            a, b = _call(R, "make_automaton"), _call(M, "make_automaton")
        # the bytes flavour of the reference returns garbage KEYS from keys()/items() (it copies its widened
        # 16-bit letters as if they were bytes: tests/test_basic.py:54-76 is an xfail "fails everywhere"),
        # so only values() can be compared there
        elif op == "keys":
            name = "keys" if fl == "unicode" else "values"
            a, b = _call(R, name), _call(M, name)
        elif op == "keys_prefix":
            name = "keys" if fl == "unicode" else "values"
            a, b = _call(R, name, w), _call(M, name, w)
        elif op == "items":
            name = "items" if fl == "unicode" else "values"
            a, b = _call(R, name), _call(M, name)
        elif op == "contains":
            a, b = ("ok", w in R), ("ok", w in M)
        else:
            a, b = _call(R, op, w), _call(M, op, w)
        assert a == b, (step, op, w, a, b)
    assert len(R) == len(M) and R.kind == M.kind


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_wildcards_stores_and_errors(fl, reference):
    ref, mine = reference(fl), ac.flavour(fl)
    c = lambda s: _conv(fl, s)  # noqa: E731
    R, M = ref.Automaton(), mine.Automaton()
    for i, w in enumerate(["he", "her", "hers", "she", "hi", "him", "his", "x", "h?r"]):
        R.add_word(c(w), i)
        M.add_word(c(w), i)
    for args in [(c("h?"), c("?")), (c("h??"), c("?")), (c("h?"), c("?"), ref.MATCH_AT_LEAST_PREFIX), (c("h??s"), c("?"), ref.MATCH_AT_MOST_PREFIX),
                 (c("h"),), (c("zz"),), (c("h?r"), c("?"), ref.MATCH_EXACT_LENGTH), (c("??"), c("?"), ref.MATCH_AT_LEAST_PREFIX)]:
        margs = tuple(getattr(mine, "MATCH_EXACT_LENGTH") if a is ref.MATCH_EXACT_LENGTH and isinstance(a, int) and False else a for a in args)
        for name in (("keys", "values", "items") if fl == "unicode" else ("values",)):
            assert _call(R, name, *args) == _call(M, name, *margs), (name, args)
    # STORE_INTS / STORE_LENGTH value rules (src/Automaton.c:225-247) and constructor validation (:20-70)
    for store in (ref.STORE_INTS, ref.STORE_LENGTH):
        R, M = ref.Automaton(store), mine.Automaton(store)
        for w in ["a", "ab", "a", "abc"]:
            assert _call(R, "add_word", c(w)) == _call(M, "add_word", c(w))
        if store == ref.STORE_INTS:
            assert _call(R, "add_word", c("zz"), 77) == _call(M, "add_word", c("zz"), 77)
            assert _call(R, "add_word", c("zy"), "no") == _call(M, "add_word", c("zy"), "no")
        assert _call(R, "values") == _call(M, "values")
        assert R.store == M.store
    assert _call(ref, "Automaton", -42) == _call(mine, "Automaton", -42)
    assert _call(ref, "Automaton", ref.STORE_ANY, -42) == _call(mine, "Automaton", mine.STORE_ANY, -42)
    assert _call(ref.Automaton(), "add_word", c("k")) == _call(mine.Automaton(), "add_word", c("k"))      # value required
    wrong = "text" if fl == "bytes" else b"text"
    for name in ("add_word", "exists", "match", "get", "longest_prefix", "remove_word"):
        args = (wrong, 1) if name == "add_word" else (wrong,)
        Rw, Mw = ref.Automaton(), mine.Automaton()
        Rw.add_word(c("k"), 0)
        Mw.add_word(c("k"), 0)
        assert _call(Rw, name, *args) == _call(Mw, name, *args), name
    # stale iterators (src/AutomatonItemsIter.c version check)
    R, M = ref.Automaton(), mine.Automaton()
    for A in (R, M):
        A.add_word(c("a"), 1)
        A.add_word(c("b"), 2)
    for A in (R, M):
        it = A.keys()
        next(it)
        A.add_word(c("new"), 3)
        with pytest.raises(ValueError):
            next(it)


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_get_stats_counts_the_letter_trie_like_the_reference(fl, reference):
    """nodes / links / words / longest_word of get_stats() (src/Automaton.c:1044-1097) after random add_word /
    remove_word / make_automaton / clear -- also for 4-byte letters, where the host arena holds one node per byte"""
    ref, mod = reference(fl), ac.flavour(fl)
    rng = np.random.default_rng(77)
    al = "ab\u0142\U0001f600" if fl == "unicode" else "abc"

    def word():
        s = "".join(al[int(j)] for j in rng.integers(0, len(al), size=int(rng.integers(1, 7))))
        return s.encode() if fl == "bytes" else s

    for _ in range(120):
        A, R = mod.Automaton(), ref.Automaton()
        ws = [word() for _ in range(int(rng.integers(0, 10)))]
        for i, w in enumerate(ws):
            A.add_word(w, i), R.add_word(w, i)
        for w in ws[::3]:
            assert A.remove_word(w) == R.remove_word(w)
        if rng.integers(0, 2) and len(R):
            A.make_automaton(), R.make_automaton()
        if rng.integers(0, 6) == 0:
            A.clear(), R.clear()
        a, r = A.get_stats(), R.get_stats()
        assert sorted(a) == sorted(r)
        for k in ("nodes_count", "words_count", "longest_word", "links_count"):
            assert a[k] == r[k], (k, ws)


def _mask_padding(chunks, letter_width):
    """node records of a pickle (src/Automaton_pickle.c:128-188) with the three padding bytes of every node header
    zeroed: the reference dumps its structs raw, uninitialised padding included"""
    out = []
    for ch in chunks:
        b = bytearray(ch)
        pos = 8                                       # a chunk starts with its node count
        while pos + 24 <= len(b):
            n = int.from_bytes(b[pos + 16:pos + 20], "little")
            b[pos + 21:pos + 24] = b"\0\0\0"
            pos += 24 + n * (letter_width + 8)
        out.append(bytes(b))
    return out


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_enumeration_order_and_pickle_records_after_removals(fl, reference):
    """keys() / values() / items() in the reference's order (a pre-order walk that takes the most recently linked child
    first, src/AutomatonItemsIter.c:125-288) and __reduce__ records identical to the reference's (pre-order, children in
    link order, src/trie.c:197-213) -- also after remove_word and re-adding, when a re-made link goes to the END of its
    parent's child array in the reference (src/trie.c:66-136, src/trienode.c:125-147)"""
    from pyahocorasick_b200 import serialize
    ref, mod = reference(fl), ac.flavour(fl)
    rng = np.random.default_rng(2026)
    al = "ab\u0142\U0001f600" if fl == "unicode" else "abcd"
    for trial in range(150):
        R, A = ref.Automaton(), mod.Automaton()
        live = []
        for _ in range(int(rng.integers(1, 30))):
            if live and rng.integers(0, 3) == 0:
                k = live.pop(int(rng.integers(0, len(live))))
                assert R.remove_word(k) == A.remove_word(k)
            else:
                w = "".join(al[int(j)] for j in rng.integers(0, len(al), size=int(rng.integers(1, 6))))
                k = w.encode() if fl == "bytes" else w
                v = int(rng.integers(0, 1000))
                R.add_word(k, v), A.add_word(k, v)
                if k not in live:
                    live.append(k)
        if trial % 2:
            R.make_automaton(), A.make_automaton()
        assert list(R.values()) == list(A.values())
        if fl == "unicode":                               # the bytes build of the reference mangles the keys it returns
            assert list(R.keys()) == list(A.keys()) and list(R.items()) == list(A.items())
        if not live:
            continue
        pr, pa = R.__reduce__()[1], serialize.reduce_args(A)
        lw = 4 if fl == "unicode" else 2
        assert _mask_padding(pr[0], lw) == _mask_padding(pa[0], lw)
        assert tuple(pr[1:]) == tuple(pa[1:])
