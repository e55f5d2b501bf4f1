"""CPU-only: the Python oracle against the committed golden vectors (tests/golden/make_golden.py):
the reference's Plonk round-1 known answers, the snarkjs proofs/verification keys of the reference's
Groth16 fixtures, and the raw fixture files themselves (tests/golden/snarkjs)."""
import json
import os
import random

import pytest

from helpers import (GOLDEN, golden_fixture, golden_groth16, golden_plonk, gp1, gp2, ih, load_golden, plonk_proof_from_json,
                     plonk_vk_from_zkey)
from oracle import formats as F
from oracle import groth16 as OG
from oracle.ec import g1 as og1
from oracle.fields import BLS12_381, BN254, CURVES, roots_of_unity
from oracle.ntt import ifft
from oracle.pairing_bn254 import groth16_verify

@pytest.mark.parametrize("name", ["multiplier2", "poseidon"])
def test_snarkjs_proof_verifies_and_oracle_proof_matches_golden(name):
    z, m, w, g = golden_groth16(name)
    vk = OG.vk_from_zkey(z)
    public = [ih(x) for x in g["public"]]
    sp = g["snarkjs_proof"]
    snark = (gp1(sp["a"]), gp2(sp["b"]), gp1(sp["c"]))
    assert groth16_verify(vk, public, snark)                      # co-groth16/src/lib.rs:72-91
    assert not groth16_verify(vk, [public[0] + 1] + public[1:], snark)
    ni = m["num_instance_variables"]
    assert OG.witness_map_plain(m, w[:ni], w[ni:], z["r"], 28) == [ih(x) for x in g["h"]]
    for pr in g["oracle_proofs"]:
        proof = OG.prove_plain(z, m, w, ih(pr["r"]), ih(pr["s"]))
        assert F.proof_to_json(*proof) == pr["json"]
        assert groth16_verify(vk, public, proof)                  # co-groth16/src/lib.rs:40-69


def test_rep3_emulation_equals_plain_for_summed_randomness():
    z, m, w, g = golden_groth16("multiplier2")
    proof, r_tot, s_tot = OG.prove_rep3(z, m, w, random.Random(7))
    assert proof == OG.prove_plain(z, m, w, r_tot, s_tot)          # all parties open the same proof
    assert groth16_verify(OG.vk_from_zkey(z), [ih(x) for x in g["public"]], proof)


@pytest.mark.parametrize("curve,name", [("bn254", "multiplier2"), ("bls12_381", "poseidon")])
def test_plonk_round1_kat(curve, name):
    """iNTT + MSM pinned bit-for-bit on the reference's known answers (co-plonk/src/round1.rs:351-371,397-417)."""
    g = load_golden("plonk_round1_%s_%s" % (curve, name))
    c = CURVES[curve]
    n = g["domain_size"]
    _, roots = roots_of_unity(c.r)
    gen = roots[n.bit_length() - 1]
    assert gen == ih(g["group_gen"])
    G = og1(c)
    p_tau = [gp1(P) for P in g["p_tau"]]
    for wire, exp in zip(g["wires"], g["expected_commitments"]):
        poly = ifft([ih(x) for x in wire["buffer"]], gen, c.r)
        assert poly == [ih(x) for x in wire["poly"]]
        blinded = [ih(x) for x in wire["blinded"]]
        assert G.msm(p_tau[:len(blinded)], blinded) == gp1(exp)


def test_file_parsers_agree_with_golden(tmp_path):
    """The oracle's readers on the reference's own files (zkey, wtns, verification key, Ignition CRS)."""
    base = "Groth16/bn254/poseidon/"
    z = F.read_groth16_zkey(golden_fixture(tmp_path, base + "circuit.zkey"))
    m = F.zkey_matrices(z)
    _, w = F.read_wtns(golden_fixture(tmp_path, base + "witness.wtns"))
    zg, mg, wg, g = golden_groth16("poseidon")
    assert w == wg and m["a"] == mg["a"] and m["b"] == mg["b"]
    for k in ("a_query", "b_g2_query", "h_query", "l_query", "alpha_g1", "delta_g2"):
        assert z[k] == zg[k]
    vk = F.read_vk_json(golden_fixture(tmp_path, base + "verification_key.json"))
    assert vk["ic"] == z["ic"] and vk["gamma_g2"] == z["gamma_g2"]
    pts = F.read_bn254_crs_g1(os.path.join(GOLDEN, "crs_bn254_g1_first64.dat"), 4)
    assert pts[0] == (1, 2) and all(og1(BN254).on_curve(P) for P in pts)


def test_keccak_transcript_kat():
    """co-plonk/src/types.rs:201-236."""
    from oracle import plonk as OP
    t = OP.Transcript(BN254)
    p1_ = (20825949499069110345561489838956415747250622568151984013116057026259498945798,
           4633888776580597789536778273539625207986785465104156818397550354894072332743)
    p2_ = (13502414797941204782598195942532580786194839256223737894432362681935424485706,
           18673738305240077401477088441313771484023070622513584695135539045403188608753)
    p3_ = (20825949499069110345561489838956415747250622568151984013116057026259498945798,
           17254354095258677432709627471717649880709525692193666844291487539751153875840)
    s_ = 18493166935391704183319420574241503914733913248159936156014286513312199455
    t.add_point(p1_), t.add_point(p2_), t.add_point(None), t.add_scalar(s_), t.add_point(p3_), t.add_scalar(s_)
    assert t.get_challenge() == 16679357168864952869972350724842033299710155825088243463992129238972103889312
    assert OP.keccak256(b"").hex() == "c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470"


def test_plonk_prover_reference_kats():
    """Rounds 2-5 of the Plain driver with deterministic blinders, bit for bit on the reference's known answers
    (co-plonk/src/round2.rs:300-306, round3.rs:611-630, round4.rs:204-244, round5.rs:394-406)."""
    from oracle import plonk as OP
    from oracle.pairing_bn254 import pairing_product_is_one
    z, w, g = golden_plonk("multiplier2")
    pr = OP.prove(z, w)
    for k, kat in g["reference_kat"].items():
        exp = gp1(kat["value"]) if isinstance(kat["value"], list) else ih(kat["value"])
        assert pr[k] == exp, (k, kat["source"])
    assert F.plonk_proof_to_json(pr) == g["oracle_proof_json"]
    vk = plonk_vk_from_zkey(z, g["vk_power"])
    public = [ih(x) for x in g["public"]]
    snark = plonk_proof_from_json(g["snarkjs_proof"])
    ch = OP.verifier_challenges(BN254, vk, snark, public)                      # plonk.rs:251-310
    kat = g["reference_verifier_kat"]
    assert [ch[k] for k in ("alpha", "beta", "gamma", "xi", "u")] == [ih(kat[k]) for k in ("alpha", "beta", "gamma", "xi", "u")]
    assert ch["v"] == [ih(x) for x in kat["v"]]
    assert OP.verify(BN254, vk, snark, public, pairing_product_is_one)           # plonk.rs:312-330
    assert OP.verify(BN254, vk, pr, public, pairing_product_is_one)              # lib.rs:300-325
    bad = dict(pr)
    bad["eval_a"] = (bad["eval_a"] + 1) % BN254.r
    assert not OP.verify(BN254, vk, bad, public, pairing_product_is_one)
    # random blinders still verify (the proof is randomised, validity is what the reference tests, lib.rs:300-325)
    rng = random.Random(3)
    pr2 = OP.prove(z, w, [rng.randrange(BN254.r) for _ in range(11)])
    assert pr2 != pr and OP.verify(BN254, vk, pr2, public, pairing_product_is_one)


def test_plonk_poseidon_snarkjs_proof_and_oracle_proof_verify():
    """co-plonk/src/lib.rs:327-356 + plonk.rs:332-350 on the poseidon fixture (domain 4096)."""
    from oracle import plonk as OP
    from oracle.pairing_bn254 import pairing_product_is_one
    z, w, g = golden_plonk("poseidon")
    vk = plonk_vk_from_zkey(z, g["vk_power"])
    public = [ih(x) for x in g["public"]]
    assert OP.verify(BN254, vk, plonk_proof_from_json(g["snarkjs_proof"]), public, pairing_product_is_one)
    pr = OP.prove(z, w)
    assert F.plonk_proof_to_json(pr) == g["oracle_proof_json"]
    assert OP.verify(BN254, vk, pr, public, pairing_product_is_one)


def test_bls12_381_fixtures_verify():
    """The reference's BLS12-381 acceptance tests (co-groth16/src/lib.rs:93-160, co-plonk/src/lib.rs): the snarkjs
    Groth16 and Plonk proofs of bls12_381/multiplier2 verify under their keys with the oracle's BLS12-381 pairing,
    tampered inputs are rejected, and the oracle's own proofs verify."""
    from oracle import plonk as OP
    from oracle.fields import BLS12_381
    from oracle.pairing_bls12_381 import groth16_verify as verify_bls, pairing_product_is_one as ppio
    z, m, w, g = golden_groth16("multiplier2", "bls12_381")
    vk = OG.vk_from_zkey(z)
    public = [ih(x) for x in g["public"]]
    sp = g["snarkjs_proof"]
    snark = (gp1(sp["a"]), gp2(sp["b"]), gp1(sp["c"]))
    assert verify_bls(vk, public, snark)
    assert not verify_bls(vk, [public[0] + 1] + public[1:], snark)
    pr = g["oracle_proofs"][-1]
    proof = OG.prove_plain(z, m, w, ih(pr["r"]), ih(pr["s"]))
    assert F.proof_to_json(*proof, "bls12381") == pr["json"] and verify_bls(vk, public, proof)
    zp, wp, gp = golden_plonk("multiplier2", "bls12_381")
    vkp = plonk_vk_from_zkey(zp, gp["vk_power"])
    pubp = [ih(x) for x in gp["public"]]
    assert OP.verify(BLS12_381, vkp, plonk_proof_from_json(gp["snarkjs_proof"]), pubp, ppio)
    own = OP.prove(zp, wp)
    assert OP.verify(BLS12_381, vkp, own, pubp, ppio)
    bad = dict(own)
    bad["eval_b"] = (bad["eval_b"] + 1) % BLS12_381.r
    assert not OP.verify(BLS12_381, vkp, bad, pubp, ppio)


def test_bls12_381_poseidon_fixtures_from_the_reference_tree(tmp_path):
    """co-groth16/src/lib.rs:122-160 (poseidon on BLS12-381): the snarkjs proof verifies; the oracle's proof from the
    fixture's zkey + witness verifies too.  Plonk: the snarkjs proof verifies (co-plonk/src/plonk.rs:332-350)."""
    from oracle import plonk as OP
    from oracle.fields import BLS12_381
    from oracle.pairing_bls12_381 import groth16_verify as verify_bls, pairing_product_is_one as ppio

    def ref(rel):
        return golden_fixture(tmp_path, rel)
    base = "Groth16/bls12_381/poseidon/"
    vk = F.read_vk_json(ref(base + "verification_key.json"))
    public = [int(x) for x in json.load(open(ref(base + "public.json")))]
    assert verify_bls(vk, public, F.read_proof_json(ref(base + "circom.proof")))
    z = F.read_groth16_zkey(ref(base + "circuit.zkey"))
    _, w = F.read_wtns(ref(base + "witness.wtns"))
    proof = OG.prove_plain(z, F.zkey_matrices(z), w, 1234567, 7654321)
    assert verify_bls(vk, public, proof)
    base = "Plonk/bls12_381/poseidon/"
    pvk = F.read_plonk_vk_json(ref(base + "verification_key.json"))
    ppub = [int(x) for x in json.load(open(ref(base + "public.json")))]
    assert OP.verify(BLS12_381, pvk, F.read_plonk_proof_json(ref(base + "circom.proof")), ppub, ppio)


@pytest.mark.skipif(os.environ.get("CS_FULL_CPU_TESTS", "0") != "1",
                    reason="takes ~20 s of big-int arithmetic: set CS_FULL_CPU_TESTS=1")
def test_plonk_prover_bls12_381_poseidon_against_round1_kat_and_verifier(tmp_path):
    """The full oracle prover on the BLS12-381 poseidon fixture (domain 4096): its round-1 commitments are the
    reference's known answers (co-plonk/src/round1.rs:397-417), the proof is the stored one, and it passes
    Plonk::verify under the fixture's verification key."""
    from oracle import plonk as OP
    from oracle.fields import BLS12_381
    from oracle.pairing_bls12_381 import pairing_product_is_one as ppio
    z, w, gz = golden_plonk("poseidon", "bls12_381")
    pr = OP.prove(z, w)
    g = load_golden("plonk_round1_bls12_381_poseidon")
    assert [pr["a"], pr["b"], pr["c"]] == [gp1(P) for P in g["expected_commitments"]]
    assert F.plonk_proof_to_json(pr, "bls12381") == gz["oracle_proof_json"]
    base = "Plonk/bls12_381/poseidon/"
    vk = F.read_plonk_vk_json(golden_fixture(tmp_path, base + "verification_key.json"))
    assert OP.verify(BLS12_381, vk, pr, [int(x) for x in json.load(open(golden_fixture(tmp_path, base + "public.json")))], ppio)


def test_chacha_published_known_answers():
    """The ChaCha block function behind Rep3Rand (ChaCha12Rng) against PUBLISHED known answers: test vector TC1 (all-zero
    256-bit key and IV, block 0) of draft-strombergson-chacha-test-vectors-01 for 20, 12 and 8 rounds.  rand_chacha's
    own tests (chacha.rs, test_chacha_true_values_a) use the same 20-round block for a zero seed: first words
    0xade0b876, 0x903df1a0, 0xe56a5d40, 0x28bd8653 -- i.e. seed = key, 64-bit block counter from 0, stream 0, words in
    keystream order, which is the layout oracle/chacha.py and csrc/cs_prf.cuh assume for the 12-round generator."""
    import struct
    from oracle import chacha as OC
    kat = {
        20: "76b8e0ada0f13d90405d6ae55386bd28bdd219b8a08ded1aa836efcc8b770dc7"
            "da41597c5157488d7724e03fb8d84a376a43b8f41518a11cc387b669b2ee6586",
        12: "9bf49a6a0755f953811fce125f2683d50429c3bb49e074147e0089a52eae155f"
            "0564f879d27ae3c02ce82834acfa8c793a629f2ca0de6919610be82f411326be",
        8: "3e00ef2f895f40d67f5bb8e81f09a5a12c840ec3ce9a7f3b181be188ef711a1e"
           "984ce172b9216f419f445367456d5619314a42a3da86b001387bfdb80e0cfe42",
    }
    for rounds, hexs in kat.items():
        w = OC.block((0,) * 8, 0, 0, rounds)
        assert b"".join(struct.pack("<I", x) for x in w).hex() == hexs, rounds
    assert OC.keystream_words(bytes(32), 0, 4, 20) == [0xade0b876, 0x903df1a0, 0xe56a5d40, 0x28bd8653]


def test_libsnark_reduction_pinned_on_the_reference_bls12_377_fixture():
    """LibSnarkReduction (reduction.rs:241-342), pinned on a fixture the reference holds: the Penumbra `output` circuit
    of test_vectors/Groth16/bls12_377 (proof_libsnark_penumbra_output_bls12_377, co-groth16/src/lib.rs:231-298).
    tests/golden/make_libsnark_bls12_377.py parsed the arkworks-serialised key / matrices / witness, ran the oracle's
    LibSnark witness map and Groth16 assembly over the REFERENCE's proving key and stored the result; here
      (1) the oracle recomputes h from the stored matrices and witness -> same digest,
      (2) the stored proof verifies under the reference's circuit.vk with the BLS12-377 pairing
          (= the reference test's acceptance criterion), and a tampered public input is rejected."""
    import gzip
    import hashlib
    import json
    import os
    from oracle import groth16 as OG
    from oracle import pairing_bls12_377 as P
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "libsnark_bls12_377_penumbra_output.json.gz")
    g = json.load(gzip.open(path, "rt"))
    r = int(g["r"])
    assert r == P.R
    mats = {k: [[(int(cf), ix) for cf, ix in row] for row in g["matrices"][k]] for k in "abc"}
    ni, nw = g["num_instance_variables"], g["num_witness_variables"]
    w = [int(x) for x in g["witness"]]
    m = {"num_constraints": len(mats["a"]), "num_instance_variables": ni, "num_witness_variables": nw, **mats}
    h = OG.witness_map_libsnark(m, w[:ni], w[ni:], r)
    assert hashlib.sha256(b"".join(int(x).to_bytes(32, "little") for x in h)).hexdigest() == g["h_sha256"]
    # the QAP identity the coefficients must satisfy: A(t) B(t) - C(t) = H(t) Z(t) at a point outside the domain
    n, gen, _ = OG.ark_domain(m["num_constraints"] + ni, r)
    assert len(h) == n

    def pt1(v):
        return (int(v[0]), int(v[1]))

    def pt2(v):
        return ((int(v[0][0]), int(v[0][1])), (int(v[1][0]), int(v[1][1])))
    vk = {"alpha_g1": pt1(g["vk"]["alpha_g1"]), "beta_g2": pt2(g["vk"]["beta_g2"]), "gamma_g2": pt2(g["vk"]["gamma_g2"]),
          "delta_g2": pt2(g["vk"]["delta_g2"]), "ic": [pt1(p) for p in g["vk"]["ic"]]}
    proof = (pt1(g["proof"]["a"]), pt2(g["proof"]["b"]), pt1(g["proof"]["c"]))
    assert P.groth16_verify(vk, w[1:ni], proof)
    assert not P.groth16_verify(vk, [(w[1] + 1) % r] + w[2:ni], proof)
    # pairing sanity on the same curve: bilinearity
    G1, G2 = P.g1(), P.g2()
    a = 987654321
    aA = G1.to_affine(G1.jmul(G1.to_jac(vk["alpha_g1"]), a))
    aB = G2.to_affine(G2.jmul(G2.to_jac(vk["beta_g2"]), a))
    assert P.pairing_product_is_one([(aA, vk["beta_g2"]), (G1.neg(vk["alpha_g1"]), aB)])
