"""The arithmetic behind the decoder's chunked avgError replay (DESIGN 4.5, k_replay_* in csrc/fic_decode.cu), as a
numpy model that runs without a GPU: above 2^24 a binary32 running sum a = A * u (u = ulp, 2^23 <= A < 2^24) that
receives an integer e = m * u + r moves to A + m + c with c = [r > u/2], or the parity of A + m on a tie r == u/2
(round to nearest even).  A run of terms therefore acts on A through its parity only -- a two-state transducer
(delta_even, delta_odd) -- and transducers compose.  The model is checked against a strictly sequential float32 sum
(FC:407 is exactly that loop); the CUDA kernels are checked against the same sum in tests/test_gpu_round2.py."""
import numpy as np
import pytest


def seq_sum(a0, terms):
    x = np.concatenate([[np.float32(a0)], terms.astype(np.float32)])
    return np.add.accumulate(x, dtype=np.float32)[-1]


def transducer(terms, sh):
    """(delta_even, delta_odd) of a run of terms on the grid u = 2^sh."""
    h = 1 << (sh - 1)
    out = []
    for p in (0, 1):
        d = 0
        for e in terms:
            e = int(e)
            m, r = e >> sh, e & ((1 << sh) - 1)
            t = p ^ (m & 1)                       # parity of A + m
            c = 1 if r > h else (t if r == h else 0)
            d += m + c
            p = t ^ c
        out.append(d)
    return out


def compose(l, r):
    """First l, then r."""
    return [l[0] + r[l[0] & 1], l[1] + r[(1 + l[1]) & 1]]


def apply(a, td, k):
    bits = np.float32(a).view(np.uint32)
    A = int(bits & 0x7FFFFF) | 0x800000
    A2 = A + td[A & 1]
    assert A2 < (1 << 24)
    return np.uint32((int(bits) & 0xFF800000) | (A2 & 0x7FFFFF)).view(np.float32)


@pytest.mark.parametrize("k", [24, 25, 27, 30])
@pytest.mark.parametrize("kind", ["ones", "odd", "small", "wide", "ties"])
def test_transducer_equals_sequential_float_sum(k, kind):
    rng = np.random.default_rng(k * 7 + len(kind))
    n = 2048
    u = 1 << (k - 23)
    if kind == "ones":
        t = np.ones(n, np.int64)
    elif kind == "odd":
        t = rng.integers(0, 50, n) * 2 + 1
    elif kind == "small":
        t = rng.integers(0, 4, n)
    elif kind == "wide":
        t = rng.integers(0, 3 * 255 * 255 + 1, n)
    else:
        t = rng.integers(0, 64, n) * u + u // 2   # every term is a tie on this grid
    for A0 in (1 << 23, (1 << 23) + 1, (1 << 23) + 12345, (3 << 22) + 7):
        a0 = np.float32(A0 * u)
        # keep the run inside the binade, as the walker's bound does
        room = ((1 << 24) - A0) * u
        cut = int(np.searchsorted(np.cumsum(t + u // 2 + 1), room))
        tt = t[:cut]
        if len(tt) == 0:
            continue
        whole = transducer(tt, k - 23)
        assert apply(a0, whole, k) == seq_sum(a0, tt)
        # composition of the halves == the whole
        mid = len(tt) // 2
        assert compose(transducer(tt[:mid], k - 23), transducer(tt[mid:], k - 23)) == whole


def test_float_sum_stalls_on_ones():
    """Why the exact prefix is only a GUESS of the binade: on a grid of 2 an added 1 is a tie that an even mantissa drops."""
    a = np.float32(1 << 24)
    assert seq_sum(a, np.ones(1000, np.int64)) == a
    assert transducer(np.ones(1000, np.int64), 1) == [0, 1]
