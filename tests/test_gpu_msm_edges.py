"""MSM edge cases on the GPU: every window size the MSM accepts, the signed-digit carry, the bucket accumulation layout, shard
slices and the glue's fixed-base windows, each compared exactly with oracle/cref.c (whose window size is arkworks' own
formula, independent of msm_pick_c) or, where n is too large for the oracle, with the closed form [sum s_i k_i] G.

The scalar families come from test_msm_digit_model.py, which checks on the CPU that they contain carry chains of every
length, chains broken by 2^(c-1) - 2 and both ends of the digit range."""
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle import cref as c
from oracle import pyref as o
from test_msm_digit_model import C_RANGE, R_MOD, adversarial_scalars, msm_nwin, msm_pick_c

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fill(rng, n, head):
    """`head` first, then uniform and circom-like scalars (bits, 32-bit values, full width) up to n"""
    out = list(head[:n])
    while len(out) < n:
        u = rng.random()
        out.append(rng.randrange(R_MOD) if u < 0.4 else rng.randrange(2) if u < 0.7 else rng.randrange(1 << 32) if u < 0.85 else rng.randrange(R_MOD))
    return out


def _mix_specials(bases, sc):
    """points at infinity and a repeated base carrying k and r - k (their terms cancel), as test_msm_g1 does"""
    bases = bases.copy()
    sc = list(sc)
    n = len(sc)
    for i in (n // 3, n - 1):
        bases[i] = 0
    j = n // 2
    bases[j + 1] = bases[j]
    sc[j + 1] = (R_MOD - sc[j]) % R_MOD
    bases[j + 2] = bases[j]
    return bases, sc


def _dot(ks, sc):
    return sum(x * y for x, y in zip(ks, sc)) % R_MOD


@pytest.fixture(scope='module')
def g1_pool():
    rng = random.Random(0x61)
    ks = [rng.randrange(1, R_MOD) for _ in range(3000)]
    return ks, c.fixed_base_g1(c.ints_to_limbs(ks))


@pytest.fixture(scope='module')
def g2_pool():
    rng = random.Random(0x62)
    ks = [rng.randrange(1, R_MOD) for _ in range(700)]
    return ks, c.fixed_base_g2(c.ints_to_limbs(ks))


def _msm_both(ctx, g2, bases, sc):
    """GPU MSM against the oracle, canonical and Montgomery scalars"""
    scl = c.ints_to_limbs(sc)
    exp = (c.msm_g2 if g2 else c.msm_g1)(bases, scl)
    run = ctx.msm_g2 if g2 else ctx.msm_g1
    assert np.array_equal(run(bases, scl), exp)
    assert np.array_equal(run(bases, c.fr_to_mont(scl), scalars_mont=True), exp)


# ------------------------------------------------------------------------------------------------ every forced window size
@pytest.mark.parametrize('cw', list(C_RANGE))
def test_forced_window_size_adversarial_scalars(ctx, monkeypatch, g1_pool, g2_pool, cw):
    monkeypatch.setenv('B2G_MSM_C', str(cw))
    rng = random.Random(cw)
    fam = adversarial_scalars(cw)
    _, bases = g1_pool
    b, sc = _mix_specials(bases, _fill(rng, len(bases), fam))
    _msm_both(ctx, False, b, sc)
    _, bases2 = g2_pool
    n2 = min(len(bases2), max(600, len(fam) + 40))
    b, sc = _mix_specials(bases2[:n2], _fill(rng, n2, fam[::-1]))
    _msm_both(ctx, True, b, sc)


# ------------------------------------------------------------------------------------------------ default window sizes at their thresholds
G1_THRESHOLDS = [(1 << 11) - 1, 1 << 11, (1 << 13) - 1, 1 << 13, (1 << 15) - 1, 1 << 15, (1 << 19) - 1, 1 << 19, (3 << 18) - 1, 3 << 18]
G2_THRESHOLDS = [1 << 11, 1 << 19, (3 << 18) - 1]


@pytest.fixture(scope='module')
def big_pool(ctx):
    rng = random.Random(0xB19)
    n = 3 << 18
    ks = [rng.randrange(1, R_MOD) for _ in range(n)]
    lim = c.ints_to_limbs(ks)
    return ks, ctx.fixed_base_g1(lim), ctx.fixed_base_g2(lim)


def test_pick_c_thresholds_cover_every_default_window():
    assert sorted({msm_pick_c(n) for n in G1_THRESHOLDS}) == [8, 11, 13, 15, 16, 17]
    assert {msm_pick_c(n) for n in G2_THRESHOLDS} == {11, 16}


@pytest.mark.parametrize('g2,n', [(False, n) for n in G1_THRESHOLDS] + [(True, n) for n in G2_THRESHOLDS])
def test_default_window_size_at_threshold_closed_form(ctx, big_pool, g2, n):
    ks, b1, b2 = big_pool
    rng = random.Random(n * 2 + g2)
    sc = _fill(rng, n, adversarial_scalars(msm_pick_c(n))[:400])
    bases = (b2 if g2 else b1)[:n]
    got = (ctx.msm_g2 if g2 else ctx.msm_g1)(bases, c.ints_to_limbs(sc))
    k = c.ints_to_limbs([_dot(ks, sc)])
    assert np.array_equal(got, (c.fixed_base_g2 if g2 else c.fixed_base_g1)(k)[0])


# ------------------------------------------------------------------------------------------------ accumulation layout
@pytest.mark.parametrize('chunk', ['1', '2', '3', '7'])
def test_g2_small_runs(ctx, monkeypatch, g2_pool, chunk):
    # tiny runs make buckets straddle many threads, including the whole-CTA fold of buckets with > 32 fragments
    monkeypatch.setenv('B2G_MSM_CHUNK_G2', chunk)
    rng = random.Random(int(chunk))
    _, bases = g2_pool
    n = 500
    b, sc = _mix_specials(bases[:n], _fill(rng, n, [1] * 150 + [2] * 90 + adversarial_scalars(12)[:60]))
    _msm_both(ctx, True, b, sc)


@pytest.mark.parametrize('g2', [False, True], ids=['g1', 'g2'])
@pytest.mark.parametrize('chunk', [64, 7])
def test_bucket_spanning_32_and_33_runs(ctx, monkeypatch, g1_pool, g2_pool, g2, chunk):
    # one bucket over exactly MSM_BIG_FRAGS runs (msm_fold) and over one more (msm_fold_big), starting on a run boundary
    # (all scalars 1: bucket 0 from position 0) and inside a run (5 scalars 1 ahead of the scalars 2 of bucket 1)
    monkeypatch.setenv('B2G_MSM_CHUNK', str(chunk))
    monkeypatch.setenv('B2G_MSM_CHUNK_G2', str(chunk))
    _, bases = (g2_pool if g2 else g1_pool)
    lead, full = 5, 32 * chunk
    for runs, sc in ((32, [1] * full), (33, [1] * (full + 1)), (32, [1] * lead + [2] * (full - lead)), (33, [1] * lead + [2] * (full - lead + 1))):
        start, end = sc.index(sc[-1]), len(sc)              # the last bucket: bucket 0 or bucket 1
        assert (end - 1) // chunk - start // chunk + 1 == runs
        reps = -(-end // len(bases))
        b = np.concatenate([bases] * reps)[:end]
        scl = c.ints_to_limbs(sc)
        exp = (c.msm_g2 if g2 else c.msm_g1)(b, scl)
        assert np.array_equal((ctx.msm_g2 if g2 else ctx.msm_g1)(b, scl), exp), (runs, end)


@pytest.mark.parametrize('g2', [False, True], ids=['g1', 'g2'])
def test_totals_at_run_and_slab_multiples(ctx, g1_pool, g2_pool, g2):
    # the entry count (one per non-zero digit; 'ones' scalars give exactly n) at a multiple of the run length (64) and of
    # the 128-run CTA slab that G1 brings in by one bulk copy, and one past it
    _, bases = (g2_pool if g2 else g1_pool)
    for total in (64 * 5, 64 * 5 + 1, 64 * 128, 64 * 128 + 1, 64 * 256, 64 * 256 + 1):
        reps = -(-total // len(bases))
        b = np.concatenate([bases] * reps)[:total]
        sc = c.ints_to_limbs([1] * total)
        exp = (c.msm_g2 if g2 else c.msm_g1)(b, sc)
        assert np.array_equal((ctx.msm_g2 if g2 else ctx.msm_g1)(b, sc), exp), total


@pytest.mark.parametrize('rchunk', ['1', '3', '64'])
def test_reduce_chunk(ctx, monkeypatch, g1_pool, g2_pool, rchunk):
    monkeypatch.setenv('B2G_MSM_REDUCE_CHUNK', rchunk)
    rng = random.Random(int(rchunk) + 50)
    for cw in ('8', '13'):
        monkeypatch.setenv('B2G_MSM_C', cw)
        _, bases = g1_pool
        b, sc = _mix_specials(bases, _fill(rng, len(bases), adversarial_scalars(int(cw))))
        _msm_both(ctx, False, b, sc)
        _, bases = g2_pool
        b, sc = _mix_specials(bases[:600], _fill(rng, 600, adversarial_scalars(int(cw))[:200]))
        _msm_both(ctx, True, b, sc)


_BULK_CHILD = r'''
import random, sys
import numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + '/tests')
from oracle import cref as c
from circom_compat_b200 import Context
from test_msm_digit_model import R_MOD, adversarial_scalars
ctx = Context(0)
rng = random.Random(7)
for g2, n in ((False, 64 * 128 + 1), (False, 3000), (True, 64 * 128), (True, 700)):
    ks = [rng.randrange(1, R_MOD) for _ in range(n)]
    b = (c.fixed_base_g2 if g2 else c.fixed_base_g1)(c.ints_to_limbs(ks))
    if n in (3000, 700):
        fam = adversarial_scalars(11)
        sc = fam + [rng.randrange(R_MOD) for _ in range(n - len(fam))]
        b[5] = 0; b[9] = b[8]
    else:
        sc = [1] * n
    sc = c.ints_to_limbs(sc)
    got = (ctx.msm_g2 if g2 else ctx.msm_g1)(b, sc)
    if not np.array_equal(got, (c.msm_g2 if g2 else c.msm_g1)(b, sc)):
        print('MISMATCH', g2, n); sys.exit(1)
ctx.close()
print('OK')
'''


@pytest.mark.parametrize('bulk', ['1', '0'])
def test_bulk_entry_slab_both_settings(bulk):
    # B2G_ACC_BULK is read once per process: '1' stages G2's entries in shared memory too, '0' turns it off for G1
    env = dict(os.environ, B2G_ACC_BULK=bulk)
    cmd = [sys.executable] + (['-s'] if sys.flags.no_user_site else []) + ['-c', _BULK_CHILD, ROOT]
    res = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and 'OK' in res.stdout, res.stdout + res.stderr


# ------------------------------------------------------------------------------------------------ whole proofs at forced window sizes
def _oracle_key(pk, cm):
    za = dict(n_vars=pk.n_vars, n_public=pk.n_public, domain_size=pk.domain_size, num_constraints=cm.num_constraints, a_csr=cm.a, b_csr=cm.b)
    for name in ('alpha_g1', 'beta_g1', 'delta_g1', 'beta_g2', 'delta_g2', 'a_query', 'b_g1_query', 'b_g2_query', 'l_query', 'h_query'):
        za[name] = np.ascontiguousarray(getattr(pk, name), dtype=np.uint64)
    return za


def _key(ctx, kind, log_n):
    from circom_compat_b200 import synth, fr_to_mont
    if kind == 'chain':
        circ, w = synth.chain_circuit(1 << log_n), synth.chain_witness(1 << log_n)
    else:
        circ, w = synth.circomlike_circuit(log_n)
    pk, _ = synth.setup(ctx, circ)
    return circ, pk, circ.matrices(), fr_to_mont(w)


@pytest.mark.parametrize('kind', ['chain', 'circomlike'])
def test_proof_at_forced_window_sizes(ctx, monkeypatch, kind):
    from circom_compat_b200 import Groth16, release
    circ, pk, cm, wm = _key(ctx, kind, 12)
    r, s = 0x5eed0123456789, 0xabcdef9876543210
    ref = c.prove(_oracle_key(pk, cm), r, s, wm)
    for cw in ('8', '12', '16', '19', '22'):
        monkeypatch.setenv('B2G_MSM_C', cw)                    # read when the key is loaded: reload it
        release(pk)
        p = Groth16.create_proof_with_reduction_and_matrices(pk, r, s, cm, circ.num_inputs, circ.num_constraints, wm, ctx)
        assert p.data == ref, cw
    release(pk); release(cm)


# ------------------------------------------------------------------------------------------------ shard slices
def _slice(total, rank, count):
    """b2g_pk_load: rank's base range [lo, lo + cnt) of a query with `total` bases"""
    lo = total * rank // count
    return lo, total * (rank + 1) // count - lo


def _sharded(pk, cm, wm, count, r, s, with_rs):
    from circom_compat_b200 import Groth16, Context
    ctxs = [Context(0, rank, count) for rank in range(count)]
    try:
        parts = [Groth16.prove_partial(pk, cm, wm, cx, r, s) if with_rs else Groth16.prove_partial(pk, cm, wm, cx) for cx in ctxs]
        return Groth16.prove_finish(pk, np.stack(parts), r, s, ctxs[-1]).data
    finally:
        for cx in ctxs:
            cx.close()


def _real_b(pk):
    """per wire 1..n_vars-1: is its B base a real point in either group"""
    b1 = np.asarray(pk.b_g1_query).reshape(pk.n_vars, -1)[1:].any(axis=1)
    b2 = np.asarray(pk.b_g2_query).reshape(pk.n_vars, -1)[1:].any(axis=1)
    return b1 | b2


def _compacted(real, lo, cnt):
    """the sparse-B rule of b2g_pk_load"""
    return cnt >= 1024 and int(real[lo:lo + cnt].sum()) * 5 < cnt * 4


@pytest.mark.parametrize('count', [2, 3, 4, 5, 8])
def test_shards_of_test_zkey(golden, test_zkey_bytes, count):
    # 3 wires: with more ranks than bases some ranks hold empty L / A / B / H slices
    from circom_compat_b200 import read_zkey, fr_to_mont, release
    pk, cm = read_zkey(test_zkey_bytes)
    g = golden['test_zkey']
    wm = fr_to_mont([int(x) for x in g['witness']])
    assert any(_slice(pk.n_vars - 1, rk, count)[1] == 0 for rk in range(count)) == (count > pk.n_vars - 1)
    for case in g['proofs']:
        for with_rs in (True, False):
            assert _sharded(pk, cm, wm, count, int(case['r']), int(case['s']), with_rs).hex() == case['proof_hex'], (count, with_rs)
    release(pk); release(cm)


@pytest.mark.parametrize('count', [2, 7])
def test_shards_of_complex_zkey(golden, complex_zkey_bytes, count):
    from circom_compat_b200 import read_zkey, fr_to_mont, release
    pk, cm = read_zkey(complex_zkey_bytes)
    g = golden['complex_zkey']
    wm = fr_to_mont(o.chain_witness(pk.n_vars, g['a']))
    for with_rs in (True, False):
        assert _sharded(pk, cm, wm, count, int(g['r']), int(g['s']), with_rs).hex() == g['proof_hex'], with_rs
    release(pk); release(cm)


def test_shards_of_sparse_b_key(ctx):
    # circom-like 2^13: every B wire is in rank 0's slice.  4 ranks: rank 0 compacted over its real bases, ranks 1-3
    # compacted to zero bases.  9 ranks: every slice is below 1024 bases, nothing is compacted and ranks 1-8 run the
    # dense path over tables that hold only points at infinity
    from circom_compat_b200 import release
    circ, pk, cm, wm = _key(ctx, 'circomlike', 13)
    real = _real_b(pk)
    total = pk.n_vars - 1
    r, s = 0x1122334455, 0x66778899
    ref = c.prove(_oracle_key(pk, cm), r, s, wm)
    sl = [_slice(total, rk, 4) for rk in range(4)]
    assert all(_compacted(real, lo, cnt) for lo, cnt in sl)
    assert real[sl[0][0]:sl[0][0] + sl[0][1]].sum() > 0 and not any(real[lo:lo + cnt].any() for lo, cnt in sl[1:])
    sl = [_slice(total, rk, 9) for rk in range(9)]
    assert not any(_compacted(real, lo, cnt) for lo, cnt in sl) and not any(real[lo:lo + cnt].any() for lo, cnt in sl[1:])
    for count in (4, 9):
        for with_rs in (True, False):
            assert _sharded(pk, cm, wm, count, r, s, with_rs) == ref, (count, with_rs)
    release(pk); release(cm)


def test_shards_with_real_b_bases_beyond_rank_0(ctx):
    # a key whose real B bases are spread over every slice (three of four B bases moved to infinity): both ranks are
    # compacted and rank 1 has to gather its scalars from its own part of the witness
    import copy
    from circom_compat_b200 import release
    circ, pk0, cm, wm = _key(ctx, 'chain', 12)
    pk = copy.copy(pk0)
    pk.b_g1_query = np.array(pk0.b_g1_query, copy=True)
    pk.b_g2_query = np.array(pk0.b_g2_query, copy=True)
    drop = np.arange(pk.n_vars) % 4 != 1
    drop[0] = False
    pk.b_g1_query[drop] = 0
    pk.b_g2_query[drop] = 0
    real = _real_b(pk)
    sl = [_slice(pk.n_vars - 1, rk, 2) for rk in range(2)]
    assert all(_compacted(real, lo, cnt) and real[lo:lo + cnt].any() for lo, cnt in sl)
    r, s = 0x4242, 0x1717
    ref = c.prove(_oracle_key(pk, cm), r, s, wm)
    for with_rs in (True, False):
        assert _sharded(pk, cm, wm, 2, r, s, with_rs) == ref, with_rs
    release(pk); release(pk0); release(cm)


def test_shards_pick_different_windows(ctx):
    # chain 2^16 at 2 ranks: slices of 32767 and 32768 bases, so the ranks run c = 13 and c = 15
    from circom_compat_b200 import release
    circ, pk, cm, wm = _key(ctx, 'chain', 16)
    sl = [_slice(pk.n_vars - 1, rk, 2) for rk in range(2)]
    assert [cnt for _, cnt in sl] == [32767, 32768] and [msm_pick_c(cnt) for _, cnt in sl] == [13, 15]
    assert not any(_compacted(_real_b(pk), lo, cnt) for lo, cnt in sl)
    r, s = 0x7777, 0x9999
    ref = c.prove(_oracle_key(pk, cm), r, s, wm)
    for with_rs in (True, False):
        assert _sharded(pk, cm, wm, 2, r, s, with_rs) == ref, with_rs
    release(pk); release(cm)


# ------------------------------------------------------------------------------------------------ glue fixed-base windows
ONES_248 = (1 << 248) - 1
BYTES_01 = int.from_bytes(b'\x01' * 32, 'little')
GLUE_RS = [(ONES_248, BYTES_01), (BYTES_01, ONES_248), (ONES_248 * pow(BYTES_01, -1, R_MOD) % R_MOD, BYTES_01),
           (BYTES_01, ONES_248 * pow(BYTES_01, -1, R_MOD) % R_MOD), ((1 << 253) - 1, (1 << 253) - 1), (ONES_248, ONES_248)]


def test_glue_windows_hit_byte_0xff(ctx, test_zkey_bytes, golden):
    # the 8-bit window tables' last entry (byte 0xff) in every product of the glue: r * delta1, r * (beta1 + b0),
    # s * delta1, s * (alpha1 + a0), s * delta2 and (r s) * delta1 (r s = 2^248 - 1 for the third and fourth pairs)
    from circom_compat_b200 import read_zkey, Groth16, fr_to_mont, release
    for r, s in GLUE_RS[2:4]:
        assert r * s % R_MOD == ONES_248
    pk, cm = read_zkey(test_zkey_bytes)
    wm = fr_to_mont([int(x) for x in golden['test_zkey']['witness']])
    za = c.zkey_arrays(test_zkey_bytes)
    for r, s in GLUE_RS:
        ref = c.prove(za, r, s, wm)
        p = Groth16.create_proof_with_reduction_and_matrices(pk, r, s, cm, cm.num_instance_variables, cm.num_constraints, wm, ctx)
        assert p.data == ref, (hex(r), hex(s))
        assert _sharded(pk, cm, wm, 2, r, s, False) == ref, (hex(r), hex(s))
    release(pk); release(cm)
    ks = sorted({k for pair in GLUE_RS for k in pair} | {ONES_248 * pow(BYTES_01, -1, R_MOD) % R_MOD * BYTES_01 % R_MOD, R_MOD - 1})
    lim = c.ints_to_limbs(ks)
    assert np.array_equal(ctx.fixed_base_g1(lim), c.fixed_base_g1(lim))
    assert np.array_equal(ctx.fixed_base_g2(lim), c.fixed_base_g2(lim))
