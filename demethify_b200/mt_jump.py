"""Jump-ahead for numpy's legacy MT19937 stream (host only).

The row-sharded bicross-validation (ic.py) needs, on every rank, only its rows of an M x N fold mask `np.random.rand(M, N) <
fraction` drawn from the global stream.  `rand` builds each double from two consecutive 32-bit words in C order, so rows [lo, hi)
are the words [2 lo N, 2 hi N) after the fold's start state.  MT19937 is linear over F2: the state J words later is p(T) applied
to the current one, with p = x^J mod phi and phi the generator's degree-19937 characteristic polynomial (Haramoto, Matsumoto,
Nishimura, Panneton, L'Ecuyer, "Efficient jump ahead for F2-linear random number generators", 2008).  Because T only shifts the
untempered word sequence, p(T) applied to the state is the XOR of the word windows x_{n+i}, i over the terms of p: a jump costs one
~20 000-word extension of the sequence plus the polynomial, which depends on J only and is cached.
"""
import functools

import numpy as np

__all__ = ["PHI_TERMS", "characteristic_polynomial", "jump_poly", "jump_state", "mask_rows"]

_N, _M = 624, 397
_DEG = 19937
_UPPER, _LOWER, _MATRIX_A = np.uint32(0x80000000), np.uint32(0x7FFFFFFF), np.uint32(0x9908B0DF)

# The exponents of phi, highest first: written by _phi_source() from characteristic_polynomial() (tests/test_mt_jump_cpu.py checks it)
PHI_TERMS = (
    19937, 19314, 19087, 18860, 18691, 18633, 18406, 18237, 18179, 18068, 17952, 17841, 17783, 17725, 17498, 17445, 17329,
    17271, 17160, 17044, 16933, 16875, 16822, 16817, 16595, 16590, 16537, 16421, 16368, 16363, 16252, 16141, 16136, 16025,
    15967, 15909, 15682, 15629, 15576, 15513, 15455, 15349, 15344, 15228, 15117, 15059, 15006, 15001, 14953, 14779, 14774,
    14721, 14605, 14552, 14547, 14436, 14325, 14320, 14209, 14151, 14093, 13866, 13813, 13760, 13697, 13639, 13533, 13528,
    13412, 13301, 13243, 13190, 13185, 13137, 12963, 12958, 12905, 12789, 12736, 12731, 12673, 12620, 12509, 12504, 12393,
    12335, 12277, 11997, 11944, 11881, 11838, 11717, 11712, 11611, 11485, 11384, 11374, 11321, 11215, 11157, 11147, 11089,
    10920, 10761, 10693, 10128, 9969, 9901, 9505, 8206, 7979, 7752, 7583, 7525, 7477, 7129, 6569, 6337, 5661, 4753, 4362, 4135,
    3908, 3681, 3454, 3227, 3000, 2773, 2493, 1870, 1643, 1585, 1416, 1189, 0)


def _extend(window, length):
    """The untempered MT19937 word sequence x_0 .. x_{length-1} that starts with the 624 words `window`
    (x_{n+624} = x_{n+397} ^ twist(upper bit of x_n | lower 31 bits of x_{n+1}))."""
    x = np.empty(max(length, _N), dtype=np.uint32)
    x[:_N] = window
    for s in range(0, length - _N, _N - _M):               # a chunk of 227 new words reads only words made before it
        n = np.arange(s, min(s + _N - _M, length - _N))
        y = (x[n] & _UPPER) | (x[n + 1] & _LOWER)
        x[n + _N] = x[n + _M] ^ (y >> np.uint32(1)) ^ np.where(y & np.uint32(1), _MATRIX_A, np.uint32(0))
    return x[:length]


def _berlekamp_massey(bits):
    """Shortest linear recurrence of a GF(2) sequence -> its characteristic polynomial as an int (bit k = coefficient of x^k)."""
    n = len(bits)
    rev = int("".join("1" if b else "0" for b in bits), 2)  # rev >> (n - 1 - t) has bit i = s_{t-i}
    c, b, L, m = 1, 1, 0, 1                                 # connection polynomial C, previous C, length, steps since the last change
    for t in range(n):
        if (c & (rev >> (n - 1 - t))).bit_count() & 1:
            prev = c
            c ^= b << m
            if 2 * L <= t:
                L, b, m = t + 1 - L, prev, 1
                continue
        m += 1
    return int(format(c, f"0{L + 1}b")[::-1], 2)           # x^L C(1/x)


def characteristic_polynomial():
    """phi from Berlekamp-Massey over 2 * 19937 bits of a seeded stream (bit 0 of the untempered words, which satisfies phi's
    recurrence from x_1 on: x_0 carries 31 bits that are not part of the state)."""
    key = np.random.RandomState(5489).get_state(legacy=True)[1]
    return _berlekamp_massey(list(_extend(key, 2 * _DEG + 1)[1:] & np.uint32(1)))


def _phi_source():
    """The PHI_TERMS constant as Python source."""
    p = characteristic_polynomial()
    return "PHI_TERMS = (" + ", ".join(str(k) for k in range(p.bit_length() - 1, -1, -1) if (p >> k) & 1) + ")"


def _square(p):
    """p(x)^2 over GF(2): bit k moves to bit 2k."""
    return int(format(p, "b").replace("", "0")[:-1] or "0", 2)


def _mod_phi(p):
    """p mod phi, with x^19937 = the lower terms of phi."""
    low = PHI_TERMS[1:]
    mask = (1 << _DEG) - 1
    while p >> _DEG:
        high, p = p >> _DEG, p & mask
        for k in low:
            p ^= high << k
    return p


@functools.lru_cache(maxsize=64)
def jump_poly(J):
    """x^J mod phi over GF(2) as an int (bit i = coefficient of x^i), one per jump distance, cached."""
    if J < 0:
        raise ValueError("negative jump")
    if J < _DEG:
        return 1 << J
    p = 1
    for bit in format(J, "b"):
        p = _mod_phi(_square(p))
        if bit == "1":
            p = _mod_phi(p << 1)
    return p


def jump_state(state, J):
    """numpy's legacy state tuple ('MT19937', key, pos, has_gauss, cached_gaussian) -> the state J 32-bit words later (a double of
    random_sample is two words).  `pos` may be anywhere in 1 .. 624 (a seeded state has 624).  The jumped state is the 624-word
    window that ends just before the next word, with pos = 1; the cached Gaussian is kept, as random_sample keeps it."""
    name, key, pos, has_gauss, gauss = state[:5]
    J = int(J)
    if J == 0:
        return state
    if not 1 <= pos <= _N:
        raise ValueError("MT19937 state position must be in 1 .. 624")
    # x_0 = key[0] and the next word is x_pos.  The new window is x_{pos+J-1} .. x_{pos+J+622}; the sequence from x_1 on
    # satisfies phi, so x_{pos+(J-1)+j} = XOR over the terms i of x^(J-1) mod phi of x_{pos+i+j}
    p = jump_poly(J - 1)
    terms = np.array([i for i, c in enumerate(reversed(format(p, "b"))) if c == "1"], dtype=np.int64)
    x = _extend(np.asarray(key, dtype=np.uint32), pos + int(terms[-1]) + _N)[pos:]
    window = np.bitwise_xor.reduce(x[terms[:, None] + np.arange(_N)[None, :]], axis=0)
    return (name, window, 1, has_gauss, gauss)


def mask_rows(state, M, N, lo, hi, fraction):
    """Rows [lo, hi) of `np.random.rand(M, N) < fraction` drawn from `state`, and the state after the whole M x N draw ->
    ((hi - lo) x N bool array, state)."""
    rs = np.random.RandomState()
    rs.set_state(jump_state(state, 2 * lo * N))
    rows = rs.random_sample((hi - lo, N)) < fraction
    return rows, jump_state(state, 2 * M * N)
