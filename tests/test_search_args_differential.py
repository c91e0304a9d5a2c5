"""iter() / find_all() argument handling against the reference extension (as recorded in tests/golden/reference), randomised: start / end (negative too),
ignore_white_space, find_all's callback form, chunked iteration with set() at random points.  The device is
the CPU emulation (tests/emul.py); what is under test is the host layer's index arithmetic and state carry-over
(src/Automaton.c:875-966, src/utils.c:293-359, src/AutomatonSearchIter.c:243-368)."""
import numpy as np
import pytest

import emul
import oracle
import pyahocorasick_b200 as pkg
from recorded_reference import reference  # noqa: F401 -- fixture

def _pair(ref, fl, rng, with_space):
    mod = pkg.flavour(fl)
    al = "abc " if with_space else "abc"

    def word(lo, hi, alphabet=al):
        s = "".join(alphabet[int(j)] for j in rng.integers(0, len(alphabet), size=int(rng.integers(lo, hi))))
        return s.encode() if fl == "bytes" else s

    keys = list(dict.fromkeys(word(1, 5, "abc") for _ in range(int(rng.integers(1, 9)))))
    A, R = mod.Automaton(), ref.Automaton()
    for i, k in enumerate(keys):
        A.add_word(k, i), R.add_word(k, i)
    A.make_automaton(), R.make_automaton()
    return A, R, word


def _call(fn, *a, **kw):
    try:
        return ("ok", list(fn(*a, **kw)))
    except Exception as e:                       # same exception type is part of the contract
        return ("exc", type(e).__name__)


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_iter_ranges_and_white_space(fl, monkeypatch, reference):
    emul.install(monkeypatch, "filter")
    rng = np.random.default_rng(21)
    for _ in range(120):
        A, R, word = _pair(reference(fl), fl, rng, with_space=True)
        hay = word(0, 30)
        n = len(hay)
        for _ in range(6):
            # iter() takes start / end as they come (:953-959): -1 means "default", any other negative start and any
            # end past the buffer make the reference read outside it -- undefined, so not part of the contract
            args = [hay]
            if rng.integers(0, 3):
                args.append(int(rng.integers(-1, n + 4)))
                if rng.integers(0, 2):
                    args.append(int(rng.integers(-1, n + 1)))
            kw = {"ignore_white_space": True} if rng.integers(0, 3) == 0 else {}
            assert _call(A.iter, *args, **kw) == _call(R.iter, *args, **kw), (fl, hay, args, kw)


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_find_all_ranges(fl, monkeypatch, reference):
    emul.install(monkeypatch, "filter")
    rng = np.random.default_rng(22)
    for _ in range(100):
        A, R, word = _pair(reference(fl), fl, rng, with_space=False)
        hay = word(0, 30)
        n = len(hay)
        for _ in range(5):
            extra = []
            if rng.integers(0, 3):
                extra.append(int(rng.integers(-n - 3, n + 4)))
                if rng.integers(0, 2):
                    extra.append(int(rng.integers(-n - 3, n + 4)))
            got, want = [], []

            def run(X, acc):
                try:
                    X.find_all(hay, lambda i, v: acc.append((i, v)), *extra)
                    return "ok"
                except Exception as e:
                    return type(e).__name__
            assert (run(A, got), got) == (run(R, want), want), (fl, hay, extra)


@pytest.mark.parametrize("ws", [False, True])
@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_iter_set_at_random_points(fl, ws, monkeypatch, reference):
    """chunks shorter than the longest key (the history then holds everything seen so far), empty chunks, extra
    next() calls past exhaustion (each moves the reference's index on by one), reset, ignore_white_space"""
    emul.install(monkeypatch, "filter")
    rng = np.random.default_rng(23 + ws)
    kw = {"ignore_white_space": True} if ws else {}
    for _ in range(150):
        A, R, word = _pair(reference(fl), fl, rng, with_space=ws)
        chunks = [word(0, 14) for _ in range(4)]
        ia, ir = A.iter(chunks[0], **kw), R.iter(chunks[0], **kw)
        got, want = [], []
        for c in chunks[1:] + [None]:
            for _ in range(int(rng.integers(0, 7))):
                for it, acc in ((ir, want), (ia, got)):
                    try:
                        acc.append(next(it))
                    except StopIteration:
                        acc.append("stop")
            if c is None:
                break
            reset = bool(rng.integers(0, 4) == 0)
            ir.set(c, reset), ia.set(c, reset)
        got += list(ia)
        want += list(ir)
        assert got == want, (fl, chunks)


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_batch_input_forms_equal_looping_the_reference(fl, monkeypatch, reference):
    """find_all_batch over a list, over (flat, offsets), over a uint8 matrix == iter() of the reference per haystack"""
    emul.install(monkeypatch, "filter")
    ref, mod = reference(fl), pkg.flavour(fl)
    rng = np.random.default_rng(31)
    al = "ab\u0142" if fl == "unicode" else "abc"

    def word(lo, hi):
        s = "".join(al[int(j)] for j in rng.integers(0, len(al), size=int(rng.integers(lo, hi))))
        return s.encode() if fl == "bytes" else s

    for _ in range(60):
        keys = list(dict.fromkeys(word(1, 6) for _ in range(int(rng.integers(1, 8)))))
        A, R = mod.Automaton(), ref.Automaton()
        for i, k in enumerate(keys):
            A.add_word(k, (i, k)), R.add_word(k, (i, k))
        A.make_automaton(), R.make_automaton()
        hays = [word(0, 20) for _ in range(int(rng.integers(0, 6)))]
        want = [(h, e, v) for h, hay in enumerate(hays) for e, v in R.iter(hay)]
        m = A.find_all_batch(hays)
        assert list(m) == want
        assert m.per_haystack(len(hays)) == [list(R.iter(h)) for h in hays]
        if fl == "bytes" and hays:
            flat = np.frombuffer(b"".join(hays), dtype=np.uint8)
            off = np.concatenate([[0], np.cumsum([len(h) for h in hays])]).astype(np.int64)
            assert list(A.find_all_batch((flat, off))) == want
            rows = rng.integers(97, 100, size=(int(rng.integers(1, 5)), int(rng.integers(1, 12))), dtype=np.uint8)
            assert list(A.find_all_batch(rows)) == [(h, e, v) for h in range(rows.shape[0]) for e, v in R.iter(rows[h].tobytes())]


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_key_sequences_iter_and_iter_long(fl, monkeypatch, reference):
    emul.install(monkeypatch, "filter")
    ref, mod = reference(fl), pkg.flavour(fl)
    rng = np.random.default_rng(32)
    vals = [0, 1, 97, 255, 256, 65535 if fl == "bytes" else 2 ** 32 - 1]
    for _ in range(80):
        keys = list({tuple(int(vals[j]) for j in rng.integers(0, len(vals), size=int(rng.integers(1, 5))))
                     for _ in range(int(rng.integers(1, 6)))})
        A, R = mod.Automaton(mod.STORE_INTS, mod.KEY_SEQUENCE), ref.Automaton(ref.STORE_INTS, ref.KEY_SEQUENCE)
        for i, k in enumerate(keys):
            A.add_word(k, i), R.add_word(k, i)
        A.make_automaton(), R.make_automaton()
        hay = tuple(int(vals[j]) for j in rng.integers(0, len(vals), size=int(rng.integers(0, 25))))
        assert list(A.iter(hay)) == list(R.iter(hay))
        assert list(A.iter_long(hay)) == list(R.iter_long(hay))


def test_streaming_over_mixed_narrow_and_wide_chunks_equals_the_oracle(monkeypatch):
    """unicode flavour, chunks that are latin-1 (scanned with the 1-byte automaton) and chunks that are not, set() at
    random points: against the C restatement (oracle/ac_oracle.c), which has no storage-kind special cases"""
    emul.install(monkeypatch, "filter")
    rng = np.random.default_rng(5)
    mod = pkg.flavour("unicode")

    def word(al, lo, hi):
        return "".join(al[int(j)] for j in rng.integers(0, len(al), size=int(rng.integers(lo, hi))))

    for _ in range(250):
        kal = ["ab\xe9", "abł", "ab\xe9ł\U0001f600"][int(rng.integers(0, 3))]
        keys = list({word(kal, 1, 6) for _ in range(int(rng.integers(1, 7)))})
        A, O = mod.Automaton(mod.STORE_INTS), oracle.OracleAutomaton()
        for i, k in enumerate(keys):
            A.add_word(k, i), O.add_word(k, i)
        A.make_automaton(), O.make_automaton()
        chunks = [word(["ab\xe9", "abł\U0001f600", "ab"][int(rng.integers(0, 3))], 0, 12) for _ in range(int(rng.integers(1, 6)))]
        ia, io = A.iter(chunks[0]), O.iter(chunks[0])
        got, want = [], []
        for ci in range(len(chunks)):
            for _ in range(int(rng.integers(0, 6))):
                for it, acc in ((io, want), (ia, got)):
                    try:
                        acc.append(next(it))
                    except StopIteration:
                        acc.append("stop")
            if ci + 1 < len(chunks):
                reset = bool(rng.integers(0, 5) == 0)
                io.set(chunks[ci + 1], reset), ia.set(chunks[ci + 1], reset)
        got += list(ia)
        want += list(io)
        assert got == want, (keys, chunks)


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_ignore_white_space_uses_the_c_library_classes(fl, monkeypatch, reference):
    """which letters count as white space is libc's business (iswspace / isspace, src/AutomatonSearchIter.c:265-270):
    control characters, NEL, no-break space, and for the unicode build the wide ones"""
    emul.install(monkeypatch, "filter")
    ref, mod = reference(fl), pkg.flavour(fl)
    rng = np.random.default_rng(9)
    ws = [" ", "\t", "\n", "\x0b", "\x0c", "\r", "\x85", "\xa0", "\x1c", "\x1f"]
    if fl == "unicode":
        ws += [" ", "　", "​", " "]
    al = list("ab") + ws

    def word(lo, hi, alphabet):
        s = "".join(alphabet[int(j)] for j in rng.integers(0, len(alphabet), size=int(rng.integers(lo, hi))))
        return s.encode("latin-1") if fl == "bytes" else s

    for _ in range(150):
        keys = list(dict.fromkeys(word(1, 5, list("ab")) for _ in range(int(rng.integers(1, 6)))))
        A, R = mod.Automaton(), ref.Automaton()
        for i, k in enumerate(keys):
            A.add_word(k, i), R.add_word(k, i)
        A.make_automaton(), R.make_automaton()
        hay = word(0, 25, al)
        assert list(A.iter(hay, ignore_white_space=True)) == list(R.iter(hay, ignore_white_space=True)), (keys, hay)


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_searches_between_random_mutations(fl, monkeypatch, reference):
    """add_word / remove_word / make_automaton in random order, searching whenever the reference can (and raising
    like it when it cannot) -- including automata from which every key has been removed again"""
    emul.install(monkeypatch, "filter")
    ref, mod = reference(fl), pkg.flavour(fl)
    rng = np.random.default_rng(13)
    al = "abc" if fl == "bytes" else "abł"

    def word(lo, hi):
        s = "".join(al[int(j)] for j in rng.integers(0, len(al), size=int(rng.integers(lo, hi))))
        return s.encode() if fl == "bytes" else s

    def outcome(X, hay):
        try:
            return list(X.iter(hay))
        except Exception as e:
            return type(e).__name__

    for _ in range(120):
        A, R = mod.Automaton(), ref.Automaton()
        first = word(1, 2)
        A.add_word(first, -1), R.add_word(first, -1)            # the reference asserts on a never-filled trie
        for _ in range(int(rng.integers(3, 25))):
            op, w = int(rng.integers(0, 10)), word(1, 6)
            if op < 5:
                v = int(rng.integers(0, 100))
                assert A.add_word(w, v) == R.add_word(w, v)
            elif op < 7:
                assert A.remove_word(w) == R.remove_word(w)
            elif op < 9:
                assert A.make_automaton() == R.make_automaton()
                if R.kind == ref.AHOCORASICK:
                    hay = word(0, 30)
                    assert list(A.iter(hay)) == list(R.iter(hay))
                    assert list(A.iter_long(hay)) == list(R.iter_long(hay))
            else:
                hay = word(0, 12)
                assert outcome(A, hay) == outcome(R, hay)
        assert len(A) == len(R) and A.kind == R.kind


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_iter_long_ranges_and_batch(fl, monkeypatch, reference):
    """iter_long(string, [start, [end]]) uses find_all's range rules (src/Automaton.c:968-1040); find_long_batch ==
    looping it.  The unicode key sets mix latin-1 and other letters over latin-1 haystacks on purpose."""
    emul.install(monkeypatch, "filter")
    ref, mod = reference(fl), pkg.flavour(fl)
    rng = np.random.default_rng(17)
    al = "abc" if fl == "bytes" else "abł"

    def word(lo, hi):
        s = "".join(al[int(j)] for j in rng.integers(0, len(al), size=int(rng.integers(lo, hi))))
        return s.encode() if fl == "bytes" else s

    for _ in range(120):
        keys = list(dict.fromkeys(word(1, 6) for _ in range(int(rng.integers(1, 8)))))
        A, R = mod.Automaton(), ref.Automaton()
        for i, k in enumerate(keys):
            A.add_word(k, i), R.add_word(k, i)
        A.make_automaton(), R.make_automaton()
        hays = [word(0, 25) for _ in range(int(rng.integers(1, 5)))]
        assert list(A.find_long_batch(hays)) == [(h, e, v) for h, hay in enumerate(hays) for e, v in R.iter_long(hay)]
        for hay in hays:
            n = len(hay)
            args = [hay]
            if rng.integers(0, 2):
                args.append(int(rng.integers(-n - 2, n + 3)))
                if rng.integers(0, 2):
                    args.append(int(rng.integers(-n - 2, n + 3)))
            assert _call(A.iter_long, *args) == _call(R.iter_long, *args), (keys, args)
