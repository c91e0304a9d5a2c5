"""AutomatonSearchIterLong.set() (src/AutomatonSearchIterLong.c:156-212) against the reference extension (as recorded):
random keys, random chunks, set() after a random number of next() calls (before a match, between matches,
after exhaustion, after extra calls past exhaustion), with and without reset.  On CPU the device is the
emulation of tests/emul.py; the gpu-marked twin runs the real ACB_ALGO_LONG kernel."""
import numpy as np
import pytest

import emul
import pyahocorasick_b200 as pkg
from recorded_reference import reference  # noqa: F401 -- fixture

def _fuzz(ref, fl, trials, seed):
    mod = pkg.flavour(fl)
    rng = np.random.default_rng(seed)
    al = "abc"

    def word(lo, hi):
        s = "".join(al[int(j)] for j in rng.integers(0, len(al), size=int(rng.integers(lo, hi))))
        return s.encode() if fl == "bytes" else s

    for _ in range(trials):
        keys = list(dict.fromkeys(word(1, 5) for _ in range(int(rng.integers(1, 8)))))
        A, R = mod.Automaton(), ref.Automaton()
        for i, k in enumerate(keys):
            A.add_word(k, i), R.add_word(k, i)
        A.make_automaton(), R.make_automaton()
        chunks = [word(0, 12) for _ in range(4)]
        ia, ir = A.iter_long(chunks[0]), R.iter_long(chunks[0])
        got, want = [], []
        for c in chunks[1:] + [None]:
            for _ in range(int(rng.integers(0, 6))):
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
        assert got == want, (fl, keys, chunks)


@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_iter_long_set_matches_the_reference_emulated(fl, monkeypatch, reference):
    emul.install(monkeypatch, "filter")
    _fuzz(reference(fl), fl, 150, 11)


@pytest.mark.gpu
@pytest.mark.parametrize("fl", ["bytes", "unicode"])
def test_iter_long_set_matches_the_reference_on_gpu(fl, reference):
    _fuzz(reference(fl), fl, 25, 12)


def test_iter_long_set_documented_example_and_errors(monkeypatch):
    """the straddling key is found, positions continue, and the argument rules are the reference's"""
    emul.install(monkeypatch, "filter")
    mod = pkg.flavour("bytes")
    A = mod.Automaton()
    for i, k in enumerate([b"he", b"here", b"her", b"abcd"]):
        A.add_word(k, i)
    A.make_automaton()
    it = A.iter_long(b"xxhe")
    assert list(it) == [(3, 0)]
    it.set(b"re is abcd")                     # the walk restarted after "he": nothing straddles
    assert list(it) == [(4 + 9, 3)]
    it.set(b"..ab")
    assert list(it) == []
    it.set(b"cd!")                            # "abcd" straddles the seam: 14 + 4 + 1
    assert list(it) == [(19, 3)]
    it.set(b"here", True)
    assert list(it) == [(3, 1)]
    with pytest.raises(IndexError):
        it.set()
    with pytest.raises(TypeError):
        it.set("text")
    A.add_word(b"zzz", 9)
    with pytest.raises(ValueError, match="has changed"):
        next(it)


def _stream_case(mod):
    A = mod.Automaton()
    for i, k in enumerate([b"abcd", b"bcdx", b"q", b"abcdefghij"]):
        A.add_word(k, i)
    A.make_automaton()
    return A


def test_iter_long_stream_uploads_only_the_new_chunk(monkeypatch):
    """a stream without matches: every set() scans its own chunk and nothing else (the walk's state travels as a
    state id, acb_table_set_long_state / acb_table_get_long_state); keys spread over many chunks are still found"""
    fake = emul.install(monkeypatch, "filter")
    sizes = []

    def counting(self, flat, *a, **kw):
        sizes.append(int(np.asarray(flat).size))
        return fake(self, flat, *a, **kw)
    from pyahocorasick_b200 import automaton as am
    monkeypatch.setattr(am.Automaton, "_scan_flat", counting)
    mod = pkg.flavour("bytes")
    A = _stream_case(mod)
    it = A.iter_long(b"z" * 100)
    assert list(it) == []
    for _ in range(50):
        it.set(b"zab" * 33 + b"z")                        # ends inside nothing; "ab" prefixes never complete
        assert list(it) == []
    assert sizes == [100] * 51
    pos = 100 * 51
    for ch in (b"a", b"b", b"c", b"d", b"e"):              # "abcd" over four chunks, reported when the walk fails on "e"... or at the end
        it.set(ch)
        got = list(it)
        pos += 1
        if ch == b"d":
            assert got == [(pos - 1, 0)]                   # end of the chunk with a pending match: reported at once
        else:
            assert got == []
    assert sizes[-5:] == [1] * 5


@pytest.mark.gpu
def test_iter_long_long_stream_on_gpu(reference):
    """the same stream through the real ACB_ALGO_LONG kernel, against the reference extension"""
    ref, mod = reference("bytes"), pkg.flavour("bytes")
    A, R = _stream_case(mod), _stream_case(ref)
    rng = np.random.default_rng(5)
    ia, ir = A.iter_long(b"z" * 100), R.iter_long(b"z" * 100)
    assert list(ia) == list(ir)
    for _ in range(200):
        n = int(rng.integers(0, 40))
        chunk = bytes(rng.choice(np.frombuffer(b"abcdxzq", dtype=np.uint8), size=n).tolist())
        ia.set(chunk), ir.set(chunk)
        assert list(ia) == list(ir)
