"""Pin the CPU oracle (oracle/ac_oracle.c) before anything trusts it.

1. against the committed golden vectors (produced by the reference itself),
2. against the compiled reference on seeded random batches, as recorded in tests/golden/reference.
"""
import numpy as np
import pytest

import oracle
from golden_driver import all_scenarios, dec
from recorded_reference import reference, reference_records  # noqa: F401 -- fixtures

STORE_INTS, STORE_LENGTH, STORE_ANY = 10, 20, 30


def _build(sc):
    A = oracle.OracleAutomaton()
    n = 0
    for key, val in sc["words"]:
        k = dec(key)
        if sc["store"] == STORE_LENGTH:
            v = len(k)
        elif val is None:
            v = len(A) + 1          # src/Automaton.c:238-243 default for STORE_INTS
        else:
            v = val
        if sc["store"] != STORE_ANY:
            v = int(np.int64(v).astype(np.int32)) if -2**63 <= v < 2**63 else v   # "ii" truncation, SURVEY A7
        A.add_word(k, v)
        n += 1
    if sc.get("make", True):
        A.make_automaton()
    return A


def _norm_range(n, args, kw):
    """iter() argument defaults: -1 means 'not given' (src/Automaton.c:881-883,950-956)."""
    start = kw.get("start", args[0] if len(args) > 0 else -1)
    end = kw.get("end", args[1] if len(args) > 1 else -1)
    if start == -1:
        start = 0
    if end == -1:
        end = n
    return start, end


SC = [s for s in all_scenarios() if not s["name"].startswith("wrong_type")]


@pytest.mark.parametrize("sc", SC, ids=[s["name"] for s in SC])
def test_oracle_matches_golden(sc):
    A = _build(sc)
    checked = 0
    for op in sc["ops"]:
        if "raises" in op:
            continue            # argument validation lives in the Python layer, not in the oracle
        kind = op["op"]
        if kind == "iter":
            hay = dec(op["hay"])
            kw = op.get("kw", {})
            s, e = _norm_range(len(hay), op.get("args", []), kw)
            iws = kw.get("ignore_white_space", False) == 1
            got = [[i, v] for i, v in A.iter(hay, s, e, iws)]
            assert got == op["expect"], (sc["name"], op)
            checked += 1
        elif kind == "iter_long":
            hay = dec(op["hay"])
            a = op.get("args", [])
            if any(x < 0 for x in a):
                continue
            s = a[0] if len(a) > 0 else 0
            e = a[1] if len(a) > 1 else len(hay)
            got = [[i, v] for i, v in A.iter_long(hay, s, e)]
            assert got == op["expect"], (sc["name"], op)
            checked += 1
        elif kind == "find_all":
            hay = dec(op["hay"])
            a = op.get("args", [])
            if any(x < 0 for x in a):
                continue        # negative-index arithmetic is pinned on the Python layer
            s = a[0] if len(a) > 0 else 0
            e = a[1] if len(a) > 1 else len(hay)
            got = [[i, v] for i, v in A.find_all(hay, s, e)]
            assert got == op["expect"], (sc["name"], op)
            checked += 1
        elif kind == "iter_set":
            a = op.get("args", [])
            init = dec(op["init"])
            it = A.iter(init, a[0] if a else 0, None)
            out = []
            if op.get("drain_first"):
                out.append([[i, v] for i, v in it])
            for chunk, reset in op["chunks"]:
                it.set(dec(chunk), bool(reset))
                out.append([[i, v] for i, v in it])
            assert out == op["expect"], (sc["name"], op)
            checked += 1
        elif kind == "iter_set_partial":
            it = A.iter(dec(op["init"]))
            out = [[list(next(it)) for _ in range(op["take"])]]
            it.set(dec(op["chunk"]), op.get("reset", False))
            out.append([[i, v] for i, v in it])
            assert out == op["expect"], (sc["name"], op)
            checked += 1
        elif kind == "kind":
            assert A.kind == op["expect"]
        elif kind == "len":
            assert len(A) == op["expect"]
    assert checked or not sc.get("make", True) or not sc["words"]


def _int_automaton(mod, keys):
    A = mod.Automaton(mod.STORE_INTS)
    for i, k in enumerate(keys):
        A.add_word(k, i)
    A.make_automaton()
    return A


@pytest.mark.parametrize("seed,alpha,nw,lens,nh,hl", [
    (1, b"ab", 30, (1, 8), 50, 300),
    (2, b"ACGT", 2000, (8, 12), 200, 150),
    (3, bytes(range(48, 58)) + bytes(range(65, 91)) + bytes(range(97, 123)), 1000, (4, 16), 400, 256),
    (4, bytes(range(256)), 500, (1, 4), 100, 1000),
])
def test_oracle_matches_reference_batch(seed, alpha, nw, lens, nh, hl, reference, reference_records):
    rng = np.random.Generator(np.random.PCG64(seed))
    al = np.frombuffer(alpha, dtype=np.uint8)
    keys = [al[rng.integers(0, len(al), size=int(rng.integers(lens[0], lens[1] + 1)))].tobytes() for _ in range(nw)]
    R = _int_automaton(reference("bytes"), keys)
    O = oracle.OracleAutomaton()
    for i, k in enumerate(keys):
        O.add_word(k, i)
    O.make_automaton()
    assert len(R) == len(O)
    assert R.get_stats()["nodes_count"] == O.nodes_count
    flat = al[rng.integers(0, len(al), size=nh * hl)]
    for h in range(nh):      # plant one key per haystack
        k = np.frombuffer(keys[int(rng.integers(0, nw))], dtype=np.uint8)
        p = int(rng.integers(0, hl - len(k)))
        flat[h * hl + p:h * hl + p + len(k)] = k
    off = np.arange(nh + 1, dtype=np.int64) * hl
    got = O.scan_batch_bytes(flat, off)
    hays = [flat[off[h]:off[h + 1]].tobytes() for h in range(nh)]
    want = reference_records("batch", lambda ref: oracle.ref_scan_batch(_int_automaton(ref, keys), hays))
    assert want.n > 0
    assert [tuple(r) for r in got.tolist()] == want      # same records, same order
