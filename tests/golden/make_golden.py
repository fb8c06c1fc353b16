"""Generates tests/golden/golden_vectors.json from a checkout of the reference, ark-circom (arkworks-rs/circom-compat):
    python tests/golden/make_golden.py <path to the ark-circom checkout>
The tests only read the JSON this writes; they never need the checkout.  Sources of every value:
  * kat_fq_one / kat_g1_one / kat_g2_one : byte vectors printed by snarkjs and pinned by the reference's own tests
    (src/zkey.rs:398-432, expectations :435-463) - extracted from that file by regex, not retyped.
  * test_zkey / complex_zkey proofs: computed by oracle/pyref.py (big-int arithmetic, independent of the C and CUDA
    code) for fixed (r, s); each proof is checked with the pairing verifier before it is written.  They equal the
    self-derived vectors of SURVEY.md App. E.
The reference never pins proof bytes (its tests use thread_rng and assert `verified`, src/zkey.rs:865-872), so these
are "oracle-derived + verifier-checked" goldens, not arkworks outputs.
"""
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, '..', '..'))
from oracle import pyref as o  # noqa: E402

REF = None                                               # the ark-circom checkout, from the command line
R = 0x1234567890abcdef1234567890abcdef
S = 0xfedcba0987654321fedcba0987654321


def rust_byte_vec(src, fn_name):
    m = re.search(r'fn %s\(\) -> Vec<u8> \{\s*vec!\[(.*?)\]' % fn_name, src, re.S)
    return [int(x) for x in re.findall(r'\d+', m.group(1))]


def deser_key_kat(src):
    """The reference's largest known-answer test, `fn deser_key` (src/zkey.rs:545-763): every point of
    test.zkey's IC / A / B1 / B2 / L / H queries as the raw bytes it feeds to deserialize_g1 / deserialize_g2.  Extracted
    by regex from that function's body (not retyped): {field: [[byte, ...] per point]}."""
    body = re.search(r'fn deser_key\(\) \{(.*?)\n    \}\n', src, re.S).group(1)
    out, pos = {}, 0
    for m in re.finditer(r'assert_eq!\(expected, params\.([a-z0-9_.]+)\);', body):
        chunk, pos = body[pos:m.start()], m.end()
        pts = []
        for kind, nums in re.findall(r'deserialize_(g1|g2)\(\s*&mut &\[(.*?)\]\[\.\.\]', chunk, re.S):
            b = [int(x) for x in re.findall(r'\d+', nums)]
            assert len(b) == (64 if kind == 'g1' else 128), (m.group(1), len(b))
            pts.append(b)
        out[m.group(1).split('.')[-1]] = pts
    assert {k: len(v) for k, v in out.items()} == {'gamma_abc_g1': 2, 'a_query': 4, 'b_g1_query': 4, 'b_g2_query': 4, 'l_query': 2, 'h_query': 4}
    return out


def field_constant_kats():
    """The scalar-field constants the reference's own sources hold as literals (SURVEY.md section 8c), by regex:
    r as the hex string its witness-calculator test asserts (src/witness/witness_calculator.rs:328-332), R^-1 mod r as the
    decimal it hard-codes (src/witness/memory.rs:45-48; R = 2^256), r as the little-endian bytes its .r1cs reader accepts
    (src/circom/r1cs_reader.rs:180-182)."""
    wc = open(os.path.join(REF, 'src/witness/witness_calculator.rs')).read()
    mem = open(os.path.join(REF, 'src/witness/memory.rs')).read()
    r1 = open(os.path.join(REF, 'src/circom/r1cs_reader.rs')).read()
    r_hex = re.search(r'wtns\.prime\.to_str_radix\(16\),\s*"([0-9A-Fa-f]{64})"', wc).group(1).lower()
    r_inv = re.search(r'let r_inv = BigInt::from_str\(\s*"(\d+)"', mem).group(1)
    r_le = re.search(r'hex::decode\("([0-9a-f]{64})"\)', r1).group(1)
    return {'r_hex': r_hex, 'r_inv_dec': r_inv, 'r_le_hex': r_le}


def witness_kats():
    """The witnesses the reference's witness-calculator tests expect (src/witness/witness_calculator.rs:260-311): multiplier_1/2/3
    (inputs test-vectors/mycircuit-input{1,2,3}.json on mycircuit.r1cs; 2 and 3 wrap around the field) by regex from the test
    source, and safe_multipler = test-vectors/safe-circuit-witness.json (circuit2, 132 wires).  Witness GENERATION is out of scope
    here; these vectors are reference-pinned INPUTS of the proving path and known-answers for the .r1cs / .wtns readers."""
    src = open(os.path.join(REF, 'src/witness/witness_calculator.rs')).read()
    mult = []
    for k in (1, 2, 3):
        body = re.search(r'async fn multiplier_%d\(\) \{(.*?)\n    \}\n' % k, src, re.S).group(1)
        wit = re.search(r'witness: &\[(.*?)\]', body, re.S).group(1)
        mult.append(re.findall(r'"(\d+)"', wit))
        assert len(mult[-1]) == 4
    inputs = [json.load(open(os.path.join(REF, 'test-vectors/mycircuit-input%d.json' % k))) for k in (1, 2, 3)]
    safe = json.load(open(os.path.join(REF, 'test-vectors/safe-circuit-witness.json')))
    return {'multiplier': mult, 'multiplier_inputs': [{k: str(v) for k, v in i.items()} for i in inputs], 'safe_multiplier': safe,
            'mycircuit_witness_json': json.load(open(os.path.join(REF, 'test-vectors/mycircuit-witness.json')))}


def main():
    out = {'r': str(R), 's': str(S)}
    src = open(os.path.join(REF, 'src/zkey.rs')).read()
    out['deser_key'] = deser_key_kat(src)
    out['kat_fq_one'] = rust_byte_vec(src, 'fq_buf')
    out['kat_g1_one'] = rust_byte_vec(src, 'g1_buf')
    out['kat_g2_one'] = rust_byte_vec(src, 'g2_buf')

    out['field_constants'] = field_constant_kats()
    out['witness_kats'] = witness_kats()

    z = o.read_zkey(open(os.path.join(HERE, 'test.zkey'), 'rb').read())
    w = [1, 33, 3, 11]                                   # test-vectors/mycircuit-witness.json
    cases = []
    for (r, s) in ((R, S), (0, S), (R, 0), (1, 1), (o.R_MOD - 1, o.R_MOD - 2)):
        A, B, C = o.prove(z, r, s, w)
        assert o.verify(z, w[1:z.num_inputs], (A, B, C))
        cases.append({'r': str(r), 's': str(s), 'proof_hex': o.proof_to_bytes(A, B, C).hex()})
    h = o.witness_map_from_matrices(z.mat_a, z.mat_b, z.num_inputs, z.num_constraints, w)
    out['test_zkey'] = {'witness': [str(x) for x in w], 'h': [str(x) for x in h], 'proofs': cases}

    z2 = o.read_zkey(open(os.path.join(HERE, 'complex-circuit-10000-10000.zkey'), 'rb').read())
    w2 = o.chain_witness(z2.n_vars, 3)                    # test-vectors/complex-circuit/input.json: a = 3
    A, B, C = o.prove(z2, R, S, w2)
    assert o.verify(z2, w2[1:z2.num_inputs], (A, B, C))
    h2 = o.witness_map_from_matrices(z2.mat_a, z2.mat_b, z2.num_inputs, z2.num_constraints, w2)
    import hashlib
    hh = hashlib.sha256(b''.join(int(x).to_bytes(32, 'little') for x in h2)).hexdigest()
    out['complex_zkey'] = {'a': 3, 'h_head': [str(x) for x in h2[:4]], 'h_sha256_canon_le': hh,
                           'proof_hex': o.proof_to_bytes(A, B, C).hex(), 'r': str(R), 's': str(S)}
    json.dump(out, open(os.path.join(HERE, 'golden_vectors.json'), 'w'), indent=1)
    print('wrote golden_vectors.json')


if __name__ == '__main__':
    if len(sys.argv) != 2 or not os.path.isfile(os.path.join(sys.argv[1], 'src', 'zkey.rs')):
        sys.exit('usage: python tests/golden/make_golden.py <path to the ark-circom checkout>')
    REF = sys.argv[1]
    main()
