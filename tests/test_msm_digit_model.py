"""Model of the MSM signed-digit decomposition in circom_compat_b200/csrc/msm.cu (CPU test, no GPU).

msm_digit_at does not walk the whole carry chain the way ark-ec 0.5 `make_digits` does: the carry into window w is read
off the windows below it (1 if the nearest window that is not exactly 2^(c-1) - 1 holds >= 2^(c-1), else 0), and the top
window never carries out.  This file restates msm_window_bits / msm_digit_at with the same 32-bit limbs, restates
make_digits with its 64-bit limbs, and checks that both give the same digits for every window size the MSM accepts
(B2G_MSM_C = 8..22), on scalar families built to contain long carry chains, broken chains and the extreme digits, plus
uniform scalars.  It pins the algorithm; tests/test_gpu_msm_edges.py runs the same families through the kernels and pins
the transcription.

The families are importable (adversarial_scalars, chain_scalars, boundary_scalars, msm_pick_c, msm_nwin) so that the GPU
tests draw the same inputs.
"""
import random

import numpy as np

R_MOD = 21888242871839275222246405745257275088548364400416034343698204186575808495617
NUM_BITS = 254                    # Fr::MODULUS_BIT_SIZE, what msm_bigint passes to make_digits
C_RANGE = range(8, 23)            # B2G_MSM_C accepts 8..22


# ------------------------------------------------------------------------------------------------ restatements
def msm_pick_c(n):
    """msm.cuh msm_pick_c: window size by base count."""
    if n >= 3 << 18:
        return 17
    if n >= 1 << 19:
        return 16
    if n >= 1 << 15:
        return 15
    if n >= 1 << 13:
        return 13
    if n >= 1 << 11:
        return 11
    lg = 0
    while (1 << (lg + 1)) <= n:
        lg += 1
    return max(8, lg - 3)


def msm_nwin(c):
    """msm.cuh msm_nwin"""
    return (255 + c - 1) // c


def limbs32(ks):
    """(N, 8) array of the 32-bit limbs of canonical scalars (held in uint64 so that shifts do not wrap)"""
    return np.array([[(k >> (32 * i)) & 0xffffffff for i in range(8)] for k in ks], dtype=np.uint64).reshape(-1, 8)


def window_bits(k32, c, w):
    """msm.cu msm_window_bits, vectorised over scalars"""
    off = w * c
    limb, sh = off >> 5, off & 31
    if limb >= 8:
        return np.zeros(len(k32), dtype=np.uint64)
    v = k32[:, limb].copy()
    if limb + 1 < 8 and sh + c > 32:
        v |= k32[:, limb + 1] << np.uint64(32)
    return (v >> np.uint64(sh)) & np.uint64((1 << c) - 1)


def digit_at(k32, c, w):
    """msm.cu msm_digit_at, vectorised over scalars: look back while the window below holds exactly 2^(c-1) - 1"""
    half = 1 << (c - 1)
    carry = np.zeros(len(k32), dtype=np.int64)
    done = np.zeros(len(k32), dtype=bool)
    for v in range(w - 1, -1, -1):
        b = window_bits(k32, c, v)
        gen = ~done & (b >= np.uint64(half))
        carry[gen] = 1
        done |= gen | (b < np.uint64(half - 1))
    coef = window_bits(k32, c, w).astype(np.int64) + carry
    cout = (coef + half) >> c
    return coef - (cout << c)


def gpu_digits(ks, c):
    """(N, nwin) digits as the kernels compute them"""
    k32 = limbs32(ks)
    return np.stack([digit_at(k32, c, w) for w in range(msm_nwin(c))], axis=1)


def make_digits(k, w, num_bits=NUM_BITS):
    """ark-ec 0.5 make_digits (variable_base/mod.rs): u64 limbs, full carry loop, the last digit keeps its carry"""
    scalar = [(k >> (64 * i)) & (2**64 - 1) for i in range(4)]
    radix = 1 << w
    mask = radix - 1
    carry = 0
    count = (num_bits + w - 1) // w
    out = []
    for i in range(count):
        bit_offset = i * w
        u64_idx, bit_idx = bit_offset // 64, bit_offset % 64
        if bit_idx < 64 - w or u64_idx == len(scalar) - 1:
            bit_buf = scalar[u64_idx] >> bit_idx
        else:
            bit_buf = (scalar[u64_idx] >> bit_idx) | ((scalar[1 + u64_idx] << (64 - bit_idx)) & (2**64 - 1))
        coef = carry + (bit_buf & mask)
        carry = (coef + radix // 2) >> w
        digit = coef - (carry << w)
        if i == count - 1:
            digit += carry << w
        out.append(digit)
    return out


# ------------------------------------------------------------------------------------------------ scalar families
def _fill_above(rng, low, shift):
    """low + (random bits above `shift`), kept below r; zero above when nothing fits"""
    room = (R_MOD - 1 - low) >> shift
    return low + (rng.randrange(room + 1) << shift if room > 0 else 0)


def chain_scalar(c, w0, run, gen, top, rng=None, broken_at=None):
    """Window w0 holds `gen` (>= 2^(c-1): it emits a carry), windows w0+1 .. w0+run hold 2^(c-1) - 1 (they pass it on),
    window w0+run+1 holds `top` and receives the carry.  broken_at = j puts 2^(c-1) - 2 in window w0+1+j instead, which
    absorbs the carry.  Random bits below w0 (all < 2^(c-1) - 1 so that nothing else carries in) and above the receiving
    window when rng is given.  Returns None if the value would not be below r."""
    half = 1 << (c - 1)
    k = gen << (c * w0)
    for j in range(run):
        k |= (half - 2 if j == broken_at else half - 1) << (c * (w0 + 1 + j))
    k |= top << (c * (w0 + run + 1))
    if rng is not None:
        for v in range(w0):
            k |= rng.randrange(half - 1) << (c * v)
    if k >= R_MOD:
        return None
    if rng is not None:
        k = _fill_above(rng, k, c * (w0 + run + 2))
    return k


def max_chain(c):
    """longest run of propagating windows (2^(c-1) - 1 above a carrying window) that fits below r"""
    run = 0
    while chain_scalar(c, 0, run + 1, 1 << (c - 1), 0) is not None:
        run += 1
    return run


def boundary_scalars(c):
    """r - 1, r - 2, (r - 1) / 2, 2^253 +- 1, 0, 1 and 2^(cw) - 1, 2^(cw), 2^(cw) + 1 at every window boundary w"""
    out = [R_MOD - 1, R_MOD - 2, (R_MOD - 1) // 2, (1 << 253) - 1, (1 << 253) + 1, 0, 1]
    for w in range(1, msm_nwin(c)):
        out += [v for v in ((1 << (c * w)) - 1, 1 << (c * w), (1 << (c * w)) + 1) if v < R_MOD]
    return out


def chain_scalars(c, seed=0):
    """Carry chains of every length up to max_chain(c), starting at the bottom window, in the middle and as high as they
    fit; the extreme carrying windows 2^(c-1) and 2^c - 1; receivers that become the top bucket (2^(c-1) - 1 with a carry
    in), the largest positive digit (2^(c-1) - 2 with a carry in) or stay small; the same chains broken by 2^(c-1) - 2."""
    rng = random.Random(seed * 1000 + c)
    half = 1 << (c - 1)
    out = []
    nwin = msm_nwin(c)
    for run in range(max_chain(c) + 1):
        starts = sorted({0, (nwin - run - 2) // 2, max(w for w in range(nwin) if chain_scalar(c, w, run, half, 0) is not None)})
        for w0 in starts:
            for gen, top, r in ((half, half - 1, None), ((1 << c) - 1, half - 2, rng), (rng.randrange(half, 1 << c), half - 1, rng),
                                (half, rng.randrange(half - 1), rng)):
                k = chain_scalar(c, w0, run, gen, top, r)
                if k is not None:
                    out.append(k)
            if run >= 1:
                for j in sorted({0, run - 1}):
                    k = chain_scalar(c, w0, run, half, half - 1, rng, broken_at=j)
                    if k is not None:
                        out.append(k)
    # top bucket without a carry: a window of exactly 2^(c-1) above a window that does not carry, at every window that fits
    for w in range(nwin):
        for below in (0, half - 2):
            k = (half << (c * w)) | ((below << (c * (w - 1))) if w else 0)
            if k < R_MOD:
                out.append(_fill_above(rng, k, c * (w + 1)))
    return out


def adversarial_scalars(c, seed=0):
    """every family above for window size c (deduplicated, order kept)"""
    seen, out = set(), []
    for k in boundary_scalars(c) + chain_scalars(c, seed):
        if k not in seen:
            seen.add(k)
            out.append(k)
    return out


# ------------------------------------------------------------------------------------------------ family census
def _windows(k, c):
    return [(k >> (c * w)) & ((1 << c) - 1) for w in range(msm_nwin(c))]


def census(ks, c):
    """What the families contain: carry-chain lengths that reach a receiving window, whether the top bucket is reached
    with and without a carry in, and whether a chain is broken by 2^(c-1) - 2."""
    half = 1 << (c - 1)
    chains, top_no_carry, top_carry, broken = set(), False, False, False
    for k in ks:
        win = _windows(k, c)
        carry_in = [0] * len(win)
        for w in range(1, len(win)):
            carry_in[w] = 1 if win[w - 1] + carry_in[w - 1] >= half else 0
        for w in range(1, len(win)):
            run = 0
            while run < w and win[w - 1 - run] == half - 1:
                run += 1
            if run < w and win[w - 1 - run] >= half:
                chains.add(run)
            if run >= 1 and run < w and win[w - 1 - run] == half - 2 and carry_in[w - 1 - run]:
                broken = True
        for w in range(len(win)):
            top_no_carry |= win[w] == half and not carry_in[w]
            top_carry |= win[w] == half - 1 and carry_in[w] == 1
    return chains, top_no_carry, top_carry, broken


# ------------------------------------------------------------------------------------------------ tests
def test_window_count_matches_make_digits():
    for c in C_RANGE:
        assert msm_nwin(c) == (NUM_BITS + c - 1) // c
        assert c * msm_nwin(c) >= NUM_BITS


def test_top_window_never_carries_out():
    # msm_digit_at drops the carry out of the top window, make_digits keeps it in the last digit: the two agree only
    # because every scalar is below r, so the top window plus a carry stays below 2^(c-1)
    for c in C_RANGE:
        top = (R_MOD - 1) >> (c * (msm_nwin(c) - 1))
        assert top + 1 < 1 << (c - 1), c


def test_families_cover_the_carry_cases():
    for c in C_RANGE:
        ks = adversarial_scalars(c)
        assert all(0 <= k < R_MOD for k in ks)
        chains, top_no_carry, top_carry, broken = census(ks, c)
        longest = max_chain(c)
        assert longest >= 3, c
        assert {1, 2, 3, longest} <= chains, (c, sorted(chains))
        assert top_no_carry and top_carry and broken, c


def _check(ks, c):
    got = gpu_digits(ks, c)
    half = 1 << (c - 1)
    assert got.min() >= -half and got.max() <= half - 1, c
    for k, row in zip(ks, got.tolist()):
        assert row == make_digits(k, c), (c, hex(k))
        assert sum(d << (c * i) for i, d in enumerate(row)) == k, (c, hex(k))


def test_digits_match_make_digits_on_families():
    for c in C_RANGE:
        ks = adversarial_scalars(c)
        _check(ks, c)
        d = gpu_digits(ks, c)
        assert (d == -(1 << (c - 1))).any() and (d == (1 << (c - 1)) - 1).any(), c     # both ends of the digit range


def test_digits_match_make_digits_on_uniform_scalars():
    rng = random.Random(0xd161)
    ks = [rng.randrange(R_MOD) for _ in range(10000)]
    for c in C_RANGE:
        _check(ks, c)


def test_chains_of_every_other_window_size_too():
    # a family built for one window size is ordinary input for the others
    ks = adversarial_scalars(8) + adversarial_scalars(13) + adversarial_scalars(17)
    for c in C_RANGE:
        _check(ks, c)
