"""The proof driver (spectre_b200/plonk.py) bound to the CPU oracle: proofs of synthetic circuits are accepted by the
independent verifier (tests/plonk_verifier.py), tampering is rejected, and the transcript layout of the
aggregation-shaped circuit is the one the reference's verifier contract hashes."""
import numpy as np
import pytest

from spectre_b200 import plonk
from spectre_b200.transcript import EvmTranscriptWrite, keccak256
from spectre_b200 import circuits as plonk_circuits
from tests import plonk_verifier
from tests.plonk_oracle_engine import OracleEngine, SeededRng


def prove(E, cs, k, fixed, advice, copies, instances, seed, digest=None):
    pk = plonk.keygen(E, cs, k, fixed, copies, vk_digest=digest)
    T = EvmTranscriptWrite(pk.vk_digest)
    proof = plonk.create_proof(E, pk, [instances], advice, SeededRng(seed), T)
    return pk, proof, T


def test_keccak_known_answers():
    assert keccak256(b"").hex() == "c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470"
    assert keccak256(b"abc").hex() == "4e03657aea45a94fc7d47ba826c8d667c0d1e6e33a64a036ec44f58fa12d6c45"


@pytest.mark.parametrize("k", [6, 8])
def test_aggregation_shape_proof_verifies(orc, k):
    cs = plonk_circuits.aggregation_shape()
    assert (cs.degree(), cs.blinding_factors(), cs.chunk_len()) == (5, 6, 3)
    instances = [11, 22, 33 + k]
    fixed, adv, copies = plonk_circuits.aggregation_witness(cs, k, instances, lookup_bits=3, groups=40)
    E = OracleEngine(k, cs.degree())
    pk, proof, T = prove(E, cs, k, fixed, [adv], copies, instances, seed=k)
    tau = orc.fr_ints(orc.srs_tau().reshape(1, 4))[0]
    assert len(proof) == 12 * 64 + 19 * 32                   # the 0x560 proof bytes of the 0x720 calldata (SURVEY.md 8: 12 points, 19 evals)
    assert plonk_verifier.verify(cs, k, pk.vk_digest, pk.fixed_commitments, pk.sigma_commitments, [instances], proof, tau)
    # any flipped evaluation or a wrong public input is rejected
    bad = bytearray(proof); bad[10 * 64 + 5] ^= 1
    with pytest.raises((AssertionError, ValueError)):
        plonk_verifier.verify(cs, k, pk.vk_digest, pk.fixed_commitments, pk.sigma_commitments, [instances], bytes(bad), tau)
    with pytest.raises(AssertionError):
        plonk_verifier.verify(cs, k, pk.vk_digest, pk.fixed_commitments, pk.sigma_commitments, [[11, 22, 34 + k]], proof, tau)


def test_unsatisfied_witness_is_rejected(orc):
    k = 6
    cs = plonk_circuits.aggregation_shape()
    instances = [5]
    fixed, adv, copies = plonk_circuits.aggregation_witness(cs, k, instances, lookup_bits=3, groups=8)
    adv[7] = plonk.fr_mont(12345)                               # break d of the second group
    E = OracleEngine(k, cs.degree())
    pk, proof, _ = prove(E, cs, k, fixed, [adv], copies, instances, seed=3)
    tau = orc.fr_ints(orc.srs_tau().reshape(1, 4))[0]
    with pytest.raises(AssertionError):
        plonk_verifier.verify(cs, k, pk.vk_digest, pk.fixed_commitments, pk.sigma_commitments, [instances], proof, tau)


def test_wide_shape_two_permutation_sets_and_theta_lookup(orc):
    k = 7
    cs = plonk_circuits.wide_shape(3)
    assert cs.degree() == 5 and len(cs.permutation) == 5
    instances = [7, 9]
    fixed, adv, copies = plonk_circuits.wide_witness(cs, k, instances, lookup_bits=3, groups=20)
    E = OracleEngine(k, cs.degree())
    pk, proof, _ = prove(E, cs, k, fixed, adv, copies, instances, seed=9)
    tau = orc.fr_ints(orc.srs_tau().reshape(1, 4))[0]
    assert plonk_verifier.verify(cs, k, pk.vk_digest, pk.fixed_commitments, pk.sigma_commitments, [instances], proof, tau)


def test_transcript_layout_matches_the_verifier_contract(kats):
    """With 14 public inputs the aggregation shape absorbs exactly the byte counts the committed contract hashes
    (tests/golden/verifier_kats.json "transcript_schedule", extracted from sync_step_verifier.sol's keccak256 calls)."""
    k = 7
    cs = plonk_circuits.aggregation_shape()
    instances = list(range(1, 15))
    fixed, adv, copies = plonk_circuits.aggregation_witness(cs, k, instances, lookup_bits=3, groups=14)
    E = OracleEngine(k, cs.degree())
    _, proof, T = prove(E, cs, k, fixed, [adv], copies, instances, seed=1)
    want = kats["transcript_schedule"]["sync_step_verifier"]
    assert T.absorbed == want["keccak_lengths"][:len(T.absorbed)]
    assert 32 * len(instances) + len(proof) == want["calldata_bytes"] and len(instances) == want["num_instances"]
    # the constants multiplying beta * x in the contract's permutation identity are DELTA and DELTA^2, in column order
    assert [int(d) for d in want["permutation_deltas"]] == [plonk.DELTA, plonk.DELTA * plonk.DELTA % plonk.R_MOD]


def _fixtures():
    import glob, os
    return sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "aggregation_k*_proof.json")))


def _contract_run(path):
    """the fixture's inputs and what the reference's verifier contract did with them: tests/golden/verifier_contract_runs.json,
    recorded by tools/extract_golden.py with tests/yul_harness.py (VK commitments substituted, pairing decided with the known tau)"""
    import json
    import os
    from tests import yul_harness
    with open(path) as f:
        fx = json.load(f)
    with open(os.path.join(os.path.dirname(__file__), "golden", "verifier_contract_runs.json")) as f:
        run = json.load(f)[os.path.basename(path)]
    contract, instances, proof, vk_points = yul_harness.fixture_inputs(fx)
    assert run["contract"] == contract and run["inputs_keccak"] == yul_harness.inputs_digest(instances, proof, vk_points), \
        "the recorded contract run is not of this fixture: re-run tools/extract_golden.py"
    return fx, run, instances, proof, vk_points


@pytest.mark.parametrize("path", _fixtures(), ids=lambda p: p.split("_")[-2])
def test_reference_verifier_contract_accepts_the_fixture(orc, path):
    """contracts/snark-verifiers/{sync_step,committee_update}_verifier.sol, interpreted as they stand in the reference tree,
    accepted the committed proofs and rejected them after a one-bit change, with a different public input, with the
    contract's own VK constants and with a wrong tau; the independent Python verifier reaches the same verdict on each."""
    from tests import plonk_verifier, yul_harness
    fx, run, instances, proof, vk_points = _contract_run(path)
    tau = orc.fr_ints(orc.srs_tau().reshape(1, 4))[0]
    assert run["verdicts"] == {"fixture": True, "flipped_evaluation_bit": False, "changed_public_input": False, "contract_vk_constants": False,
                               "wrong_tau": False}
    assert run["pairing_calls"] == 1 and run["precompile_counts"]["7"] == 21
    own = [(int(x, 16), int(y, 16)) for x, y in run["contract_vk_points"]]
    assert own[1] == vk_points[1] and own[0] != vk_points[0]      # only the range table coincides
    cs = plonk_circuits.aggregation_shape()

    def verdict(inst, prf, vk, t):
        try:
            return plonk_verifier.verify(cs, fx["k"], int(fx["vk_digest"]), vk[:4], vk[4:], [inst], prf, t)
        except (AssertionError, ValueError):
            return False
    got = {name: verdict(*case) for name, case in yul_harness.cases(instances, proof, vk_points, own, tau).items()}
    assert got == run["verdicts"]


@pytest.mark.parametrize("path", _fixtures(), ids=lambda p: p.split("_")[-2])
def test_independent_verifier_agrees_with_the_contract_term_by_term(orc, path):
    """VERDICT r1 item 8a: the independent Python verifier (tests/plonk_verifier.py) -- the check the multi-set / theta-lookup
    shapes rely on -- is pinned against the reference's verifier contract not only on accept / reject but on its intermediate
    values: every challenge it derives (theta, beta, gamma, y, x, and SHPLONK's y, v, u), x^n, the Lagrange terms l_0 and l_last,
    the instance evaluation, the quotient numerator and the expected h(x) are words the contract itself stored while verifying
    the same proof."""
    from tests import plonk_verifier
    fx, run, instances, proof, vk_points = _contract_run(path)
    assert run["verdicts"]["fixture"]
    written = {int(w, 16) for w in run["stored_words"]}
    tau = orc.fr_ints(orc.srs_tau().reshape(1, 4))[0]
    trace = {}
    cs = plonk_circuits.aggregation_shape()
    assert plonk_verifier.verify(cs, fx["k"], int(fx["vk_digest"]), vk_points[:4], vk_points[4:], [instances], proof, tau, trace=trace)
    for name in ("theta", "beta", "gamma", "y", "x", "shplonk_y", "shplonk_v", "shplonk_u", "x_n", "l_0", "l_last", "quotient_numerator", "expected_h"):
        assert trace[name] in written, "the contract never stores the verifier's %s" % name
    for q, v in trace["instance_evals"].items():
        assert v in written, "instance evaluation %r" % (q,)
    # control: a value the contract has no reason to hold is not there by accident
    assert (trace["theta"] + 1) % plonk.R_MOD not in written


def test_halo2lib_sync_step_shape_proof_verifies(orc):
    """the multi-column shape of the sync-step circuit (SURVEY.md section 8 row 1), scaled down: 4 gate columns, 2 range-lookup
    columns, the spread lookup, permutation sets of two columns"""
    k = 8
    cs = plonk_circuits.halo2lib_shape(4, 2)
    assert (cs.degree(), cs.chunk_len(), len(cs.permutation)) == (4, 2, 10)
    full = plonk_circuits.halo2lib_shape()
    assert (full.num_advice, len(full.lookups), full.degree(), len(full.permutation), -(-len(full.permutation) // full.chunk_len())) == (19, 3, 4, 21, 11)
    instances = [5, 6, 7]
    fixed, adv, copies = plonk_circuits.halo2lib_witness(cs, k, instances, lookup_bits=4, groups=30, num_gate_advice=4, num_lookup_advice=2)
    E = OracleEngine(k, cs.degree())
    pk, proof, _ = prove(E, cs, k, fixed, adv, copies, instances, seed=21)
    tau = orc.fr_ints(orc.srs_tau().reshape(1, 4))[0]
    assert plonk_verifier.verify(cs, k, pk.vk_digest, pk.fixed_commitments, pk.sigma_commitments, [instances], proof, tau)


def test_device_side_blinding_sampler_is_in_range():
    """uniform_residues (the on-device generator of the vanishing argument's random polynomial), run on torch's CPU device"""
    import torch
    g = torch.Generator().manual_seed(5)
    t = plonk.uniform_residues(torch, 50000, "cpu", g)
    a = t.numpy().view(np.uint64)
    assert a.shape == (50000, 4)
    vals = [int(r[0]) | int(r[1]) << 64 | int(r[2]) << 128 | int(r[3]) << 192 for r in a]
    assert max(vals) < plonk.R_MOD and len(set(vals)) == len(vals)
    assert 0.70 < sum(v > plonk.R_MOD // 4 for v in vals) / len(vals) < 0.80      # uniform over [0, r): three quarters above r/4


def test_lookup_violation_is_reported_like_upstream(orc):
    """an advice value outside the table makes commit_permuted fail (upstream: Error::ConstraintSystemFailure)"""
    k, instances = 7, [1]
    cs = plonk_circuits.aggregation_shape()
    fixed, adv, copies = plonk_circuits.aggregation_witness(cs, k, instances, lookup_bits=3, groups=10)
    adv[4] = plonk.fr_mont(99)
    E = OracleEngine(k, cs.degree())
    pk = plonk.keygen(E, cs, k, fixed, copies)
    with pytest.raises(ValueError):
        plonk.create_proof(E, pk, [instances], [adv], SeededRng(2), EvmTranscriptWrite(pk.vk_digest))


@pytest.mark.parametrize("variant", ["no_lookup", "no_permutation", "gates_only_negative_rotation", "two_instance_columns"])
def test_driver_edge_shapes(orc, variant):
    """constraint systems without a lookup / without a permutation, a gate reaching back with rotation -1 and a fixed query
    at rotation 1, two instance columns: proof accepted by the independent verifier"""
    from spectre_b200.plonk import Advice, Const, ConstraintSystem, Fixed, Instance, Neg, Prod, Scaled, Sum
    k = 6
    n = 1 << k
    R = plonk.R_MOD
    rows = 40
    import random
    rng = random.Random(hash(variant) & 0xffff)
    a = [rng.randrange(R) for _ in range(rows)]
    if variant == "gates_only_negative_rotation":
        # q(X) * (a(X) - 3*a(w^-1 X) - f(wX)) on rows 1..rows-1; f is a fixed column read one row ahead
        f = [0] * n
        for i in range(1, rows):
            f[i + 1] = (a[i] - 3 * a[i - 1]) % R
        q = [1 if 1 <= i < rows else 0 for i in range(n)]
        # (times a(X): cs.degree() is 3 even without a permutation -- upstream always counts permutation::Argument::required_degree() --
        # so the quotient is split into two pieces, and a degree-2 gate would leave the second one zero: a commitment to the point
        # at infinity, which the EVM transcript refuses upstream as well; see test_degree_floor_matches_upstream)
        cs = ConstraintSystem(2, 1, 0, [Prod(Prod(Fixed(0), Advice(0)), Sum(Sum(Advice(0), Neg(Scaled(Advice(0, -1), 3))), Neg(Fixed(1, 1))))], [], [])
        fixed, advice, copies, instances = [q, f], [a + [0] * (n - rows)], [], []
    elif variant == "no_lookup":
        # a * a = b with b copied from the instance column; permutation over (advice 0, advice 1, instance)
        inst = [a[i] * a[i] % R for i in range(3)]
        b = [a[i] * a[i] % R for i in range(rows)]
        q = [1 if i < rows else 0 for i in range(n)]
        cs = ConstraintSystem(1, 2, 1, [Prod(Fixed(0), Sum(Prod(Advice(0), Advice(0)), Neg(Advice(1))))], [], [("advice", 0), ("advice", 1), ("instance", 0)])
        fixed, advice, instances = [q], [a + [0] * (n - rows), b + [0] * (n - rows)], [inst]
        copies = [((1, i), (2, i)) for i in range(3)] + [((0, 5), (0, 6))]
        advice[0][6] = advice[0][5]; advice[1][6] = advice[1][5]
    elif variant == "no_permutation":
        t = 8
        table = list(range(t)) + [0] * (n - t)
        small = [rng.randrange(t) for _ in range(rows)]
        cs = ConstraintSystem(1, 1, 0, [], [([Sum(Advice(0), Const(0))], [Fixed(0)])], [])
        fixed, advice, copies, instances = [table], [small + [0] * (n - rows)], [], []
    else:
        # a + i0 = b on row 0..2, b * i1 = c; instances in two columns, both in the permutation
        i0, i1 = [rng.randrange(R) for _ in range(3)], [rng.randrange(R) for _ in range(3)]
        bcol = [0] * n; ccol = [0] * n; acol = a + [0] * (n - rows)
        x0 = [0] * n; x1 = [0] * n
        for i in range(3):
            x0[i], x1[i] = i0[i], i1[i]
            bcol[i] = (acol[i] + i0[i]) % R; ccol[i] = bcol[i] * i1[i] % R
        q = [1 if i < 3 else 0 for i in range(n)]
        cs = ConstraintSystem(1, 5, 2, [Prod(Fixed(0), Sum(Sum(Advice(0), Advice(3)), Neg(Advice(1)))), Prod(Fixed(0), Sum(Prod(Advice(1), Advice(4)), Neg(Advice(2))))], [],
                              [("advice", 3), ("advice", 4), ("instance", 0), ("instance", 1)])
        fixed, advice, instances = [q], [acol, bcol, ccol, x0, x1], [i0, i1]
        copies = [((0, i), (2, i)) for i in range(3)] + [((1, i), (3, i)) for i in range(3)]
    to_m = lambda col: np.stack([plonk.fr_mont(v) for v in col]) if len(col) else np.zeros((n, 4), np.uint64)
    E = OracleEngine(k, cs.degree())
    pk = plonk.keygen(E, cs, k, [to_m(c) for c in fixed], copies)
    T = EvmTranscriptWrite(pk.vk_digest)
    proof = plonk.create_proof(E, pk, instances, [to_m(c) for c in advice], SeededRng(7), T)
    tau = orc.fr_ints(orc.srs_tau().reshape(1, 4))[0]
    assert plonk_verifier.verify(cs, k, pk.vk_digest, pk.fixed_commitments, pk.sigma_commitments, instances, proof, tau)


def test_degree_floor_matches_upstream(orc):
    """ConstraintSystem::degree: 3 from the permutation argument even with no equality column, lookup input / table degrees
    floored at 1, minimum_degree honoured (ADVICE r1). A permutation-free degree-2 circuit therefore still has TWO quotient
    pieces; its second piece is the zero polynomial and the EVM transcript rejects the point at infinity, as upstream does."""
    from spectre_b200.plonk import Advice, Const, ConstraintSystem, Fixed, Neg, Prod, Sum
    assert ConstraintSystem(1, 1, 0, [Prod(Fixed(0), Advice(0))], [], []).degree() == 3
    assert ConstraintSystem(1, 1, 0, [], [([Const(5)], [Fixed(0)])], []).degree() == 4                       # 2 + max(1, 0) + 1
    assert ConstraintSystem(1, 2, 0, [], [([Const(5)], [Prod(Fixed(0), Prod(Advice(0), Advice(1)))])], []).degree() == 6   # 2 + 1 + 3
    assert ConstraintSystem(1, 1, 0, [Prod(Fixed(0), Advice(0))], [], [], minimum_degree=7).degree() == 7
    k = 5; n = 1 << k
    cs = ConstraintSystem(1, 1, 0, [Prod(Fixed(0), Sum(Advice(0), Neg(Advice(0))))], [], [])
    assert (cs.degree(), cs.chunk_len()) == (3, 1)
    E = OracleEngine(k, cs.degree())
    col = np.stack([plonk.fr_mont(i) for i in range(n)])
    pk = plonk.keygen(E, cs, k, [col], [])
    with pytest.raises(ValueError, match="infinity"):
        plonk.create_proof(E, pk, [], [col], SeededRng(3), EvmTranscriptWrite(pk.vk_digest))


def test_create_proof_argument_errors(orc):
    k = 6
    cs = plonk_circuits.aggregation_shape()
    fixed, adv, copies = plonk_circuits.aggregation_witness(cs, k, [1], lookup_bits=3, groups=4)
    E = OracleEngine(k, cs.degree())
    pk = plonk.keygen(E, cs, k, fixed, copies)
    new_t = lambda: EvmTranscriptWrite(pk.vk_digest)
    with pytest.raises(ValueError, match="InvalidInstances"):
        plonk.create_proof(E, pk, [], [adv], SeededRng(1), new_t())
    with pytest.raises(ValueError, match="InstanceTooLarge"):
        plonk.create_proof(E, pk, [list(range(1 << k))], [adv], SeededRng(1), new_t())
    with pytest.raises(ValueError, match="advice columns"):
        plonk.create_proof(E, pk, [[1]], [adv, adv], SeededRng(1), new_t())


def test_proving_key_file_round_trip(orc, tmp_path):
    """ProvingKey::write / ::read in upstream's RawBytesUnchecked layout (spectre_b200/plonk.py write_pk / read_pk): the key
    read back proves to the same bytes as the key it was written from, and a file for another shape is refused."""
    k, instances = 7, [3, 1, 4]
    cs = plonk_circuits.halo2lib_shape(3, 2)
    fixed, adv, copies = plonk_circuits.halo2lib_witness(cs, k, instances, lookup_bits=4, groups=20, num_gate_advice=3, num_lookup_advice=2)
    E = OracleEngine(k, cs.degree())
    pk = plonk.keygen(E, cs, k, fixed, copies)
    path = str(tmp_path / "shape.pkey")
    plonk.write_pk(E, pk, path)
    n, ext = 1 << k, 1 << E.extended_k
    nf, m = cs.num_fixed, len(cs.permutation)
    import os
    assert os.path.getsize(path) == 8 + 64 * (nf + m) + 3 * (4 + 32 * ext) + 6 * 4 + (nf + m) * (2 * (4 + 32 * n) + 4 + 32 * ext)
    pk2 = plonk.read_pk(E, cs, path)
    assert (pk2.fixed_commitments, pk2.sigma_commitments, pk2.vk_digest) == (pk.fixed_commitments, pk.sigma_commitments, pk.vk_digest)
    proofs = [plonk.create_proof(E, key, [instances], adv, SeededRng(4), EvmTranscriptWrite(key.vk_digest)) for key in (pk, pk2)]
    assert proofs[0] == proofs[1]
    with pytest.raises(ValueError):
        plonk.read_pk(E, plonk_circuits.aggregation_shape(), path)


def test_program_emits_identical_calculations_once(orc):
    """GraphEvaluator::add_calculation ([UPSTREAM] plonk/evaluation.rs) returns the existing intermediate for a repeated
    calculation; the flat program does the same (ADVICE r1), so wide gate sets do not multiply the per-row scratch. The
    value of the program is unchanged: checked against direct evaluation of the gates at every row."""
    from spectre_b200.plonk import Advice, ConstraintSystem, Fixed, Prod, Sum, Scaled
    shared = Prod(Advice(0), Advice(1, 1))
    gates = [Prod(Fixed(0), Sum(shared, Advice(2))), Prod(Fixed(0), Sum(shared, Scaled(Advice(2), 5))), Prod(Fixed(0), Sum(shared, Advice(2)))]
    cs = ConstraintSystem(1, 3, 0, gates, [], [])
    p = cs.gates_program()
    # shared product, a2*5, two distinct sums, two distinct gate products, one Horner: 7 (12 without the reuse)
    assert p["ncalc"] == 7
    n = 16
    cols = [orc.fr_random_chacha(n, 40 + i) for i in range(4)]
    y = orc.fr_random_chacha(1, 50)[0]
    zero = np.zeros(4, np.uint64)
    bgty = np.stack([zero, zero, zero, y])                       # beta, gamma, theta, y
    got = orc.graph_evaluate(p["prog"], p["ncalc"], p["ncalc"], p["constants"], p["rotations"], [cols[0]], cols[1:], [], np.zeros((1, 4), np.uint64), bgty,
                             np.zeros((n, 4), np.uint64), 1)
    R = orc.R_MOD
    f, a0, a1, a2 = [orc.fr_ints(c) for c in cols]
    yv = orc.fr_ints(y.reshape(1, 4))[0]
    for i in range(n):
        sh = a0[i] * a1[(i + 1) % n] % R
        g = [f[i] * (sh + a2[i]) % R, f[i] * (sh + 5 * a2[i]) % R, f[i] * (sh + a2[i]) % R]
        want = 0
        for v in g:
            want = (want * yv + v) % R
        assert orc.fr_ints(got[i:i + 1])[0] == want
