"""Planted near-duplicates for the matcher's second-distance recovery (match_tc.cu).  The distance kernel keeps only the
best value of each candidate set (8 trains of one parity in a 16-column group) and of each lane (queries x + 128 i) in its hot
loop; tc_resolve rebuilds the exact second distance from the winning set or lane.  Each case puts the true second neighbour
inside the winning set or lane, so the ratio test flips if that refinement is missing; the controls put it in another set."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _flip(rng, row, m):
    """row with exactly m distinct bits flipped: Hamming distance m from row."""
    bits = np.unpackbits(row)
    bits[rng.choice(256, m, replace=False)] ^= 1
    return np.packbits(bits)


def _plant(n1, n2, kind):
    rng = np.random.default_rng(n1 * 31 + n2 + len(kind))
    d1, d2 = rng.integers(0, 256, (n1, 32), dtype=np.uint8), rng.integers(0, 256, (n2, 32), dtype=np.uint8)
    mixed = kind == "mixed"
    if kind.startswith("set") or mixed:
        # query 2i + 1 at 10 bits from train j, the runner-up 1, 2 or 4 bits farther at j + step
        step = {"set1": 1, "set16": 16}.get(kind, 2)
        for i in range(min(n1 // 2, (n2 // 2 if mixed else n2) // 32)):
            j = 32 * i + int(rng.integers(0, 16 - step if step < 16 else 16))
            x = 2 * i + 1
            d1[x] = _flip(rng, d2[j], 10)
            d2[j + step] = d2[j] if kind == "setdup" else _flip(rng, d1[x], 10 + int(rng.choice([1, 2, 4])))
    if kind.startswith("lane") or mixed:
        # train y at 10 bits from query x (lane x, first tile), the runner-up 1, 2 or 4 bits farther at x + 128 k: the next
        # tile ("lane") or the last one
        y0 = n2 // 2 if mixed else 0
        for i in range(min(64, n2 - y0)):
            x, y = 2 * i, y0 + i
            k = 1 if kind == "lane" else (n1 - 1 - x) // 128
            d2[y] = _flip(rng, d1[x], 10)
            d1[x + 128 * k] = _flip(rng, d2[y], 10 + int(rng.choice([1, 2, 4])))
    return d1, d2


@pytest.mark.parametrize("n1,n2,kind", [
    (2000, 2000, "set2"), (2000, 2000, "set1"), (2000, 2000, "set16"), (2000, 2000, "setdup"), (512, 600, "lane"),
    (1000, 700, "lanek"), (1000, 777, "mixed"), (700, 2000, "mixed"), (65535, 300, "lanek")])
def test_match_planted_second(engine, oracle, n1, n2, kind):
    d1, d2 = _plant(n1, n2, kind)
    for nnr in (0.75, 0.9, 1.25):   # above 1 an exact tie passes the ratio test: lowest index wins
        for best_lr in (True, False):
            n_ref, ref = oracle.match(d1, d2, nnr, best_lr)
            n, m = engine.match(d1, d2, nnr, best_lr)
            np.testing.assert_array_equal(m, ref, err_msg=f"nnr {nnr} best_lr {best_lr}")
            assert n == n_ref
