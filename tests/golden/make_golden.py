"""Generates the golden fixtures under tests/golden/ from the reference's own test vectors.

Run once in the build container (needs /root/reference, which does not exist on the GPU box):
    python tests/golden/make_golden.py
Inputs : /root/reference/test_vectors/{Groth16,Plonk}/... and co-noir-common/src/crs/bn254_g1.dat
Expected values:
  * Plonk round-1 commitments are the REFERENCE'S known answers, typed in from
    co-circom/co-plonk/src/round1.rs:351-371 (BN254 multiplier2) and :397-417 (BLS12-381 poseidon);
    they pin iNTT + MSM bit-for-bit.
  * Groth16: the snarkjs proof / verification key / public inputs of the fixture (validity pin, the
    same criterion as co-groth16/src/lib.rs:40-91) and the oracle's proof for fixed (r, s), which this
    script first checks with the pairing verifier against that verification key.
All integers are stored as hex strings, canonical (non-Montgomery) form.
"""
import gzip
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import formats as F  # noqa: E402
from oracle import groth16 as OG  # noqa: E402
from oracle.fields import roots_of_unity  # noqa: E402
from oracle.ntt import ifft  # noqa: E402
from oracle.pairing_bn254 import groth16_verify as groth16_verify_bn254  # noqa: E402
from oracle.plonk_round1 import round1_commitments  # noqa: E402

REF = "/root/reference"


def hx(v):
    return None if v is None else format(int(v), "x")


def p1(P):
    return None if P is None else [hx(P[0]), hx(P[1])]


def p2(P):
    return None if P is None else [[hx(P[0][0]), hx(P[0][1])], [hx(P[1][0]), hx(P[1][1])]]


def dump(name, obj, compress=False):
    path = os.path.join(HERE, name + (".json.gz" if compress else ".json"))
    data = json.dumps(obj, separators=(",", ":")).encode()
    if compress:
        with gzip.GzipFile(path, "wb", mtime=0) as f:
            f.write(data)
    else:
        with open(path, "wb") as f:
            f.write(data)
    print(path, os.path.getsize(path))


def compact_plonk_key(obj, p_tau_from=None):
    """Shrinks a large Plonk key to what helpers.load_golden rebuilds it from: the selectors' evaluations over the
    domain, the permutation as indices (i -> w^i, n + i -> k1 w^i, 2n + i -> k2 w^i), no Lagrange polynomials, and
    optionally the p_tau points by reference to another fixture that holds the same ones."""
    from oracle.fields import CURVES
    r, n = CURVES[obj["curve"]].r, obj["domain_size"]
    _, roots = roots_of_unity(r)
    w = [1]
    for _ in range(n - 1):
        w.append(w[-1] * roots[n.bit_length() - 1] % r)
    index = {hx(k * x % r): j * n + i for j, k in enumerate((1, int(obj["k1"], 16), int(obj["k2"], 16))) for i, x in enumerate(w)}
    obj["q_domain_evals"] = {k: obj.pop(k)["evals"][0::4] for k in ("qm", "ql", "qr", "qo", "qc")}
    obj["sigma"] = [[index[x] for x in obj.pop(k)["evals"][0::4]] for k in ("s1", "s2", "s3")]
    del obj["lagrange"]
    if p_tau_from:
        assert load(p_tau_from)["p_tau"] == obj.pop("p_tau")
        obj["p_tau_from"] = p_tau_from
    return obj


def compact_round1(obj, blinders):
    """Drops each wire's polynomial and blinded polynomial: helpers.load_golden recomputes them from the wire values
    and the blinders (the same steps as plonk_fixture)."""
    for wire, blind in zip(obj["wires"], blinders):
        del wire["poly"], wire["blinded"]
        wire["blinders"] = blind
    return obj


def load(name):
    p = os.path.join(HERE, name + ".json")
    return json.load(gzip.open(p + ".gz") if not os.path.exists(p) else open(p))


def groth16_fixture(name, r_s_list, compress, curve_dir="bn254"):
    groth16_verify = groth16_verify_bn254
    if curve_dir == "bls12_381":
        from oracle.pairing_bls12_381 import groth16_verify
    base = "%s/test_vectors/Groth16/%s/%s/" % (REF, curve_dir, name)
    z = F.read_groth16_zkey(base + "circuit.zkey")
    m = F.zkey_matrices(z)
    _, w = F.read_wtns(base + "witness.wtns")
    vk = F.read_vk_json(base + "verification_key.json")
    pub = [int(x) for x in json.load(open(base + "public.json"))]
    sp = F.read_proof_json(base + "circom.proof")
    assert groth16_verify(vk, pub, sp), "snarkjs proof must verify"
    proofs = []
    for r_, s_ in r_s_list:
        pr = OG.prove_plain(z, m, w, r_, s_)
        assert groth16_verify(vk, pub, pr), "oracle proof must verify"
        proofs.append(dict(r=hx(r_), s=hx(s_), a=p1(pr[0]), b=p2(pr[1]), c=p1(pr[2]),
                           json=F.proof_to_json(*pr, "bn128" if curve_dir == "bn254" else "bls12381")))
    ni = m["num_instance_variables"]
    h = OG.witness_map_plain(m, w[:ni], w[ni:], z["r"], z["curve"].two_adicity)
    obj = dict(
        source="test_vectors/Groth16/%s/%s" % (curve_dir, name), curve=curve_dir,
        n_vars=z["n_vars"], n_public=z["n_public"], domain_size=z["domain_size"],
        num_constraints=m["num_constraints"], num_instance_variables=ni,
        num_witness_variables=m["num_witness_variables"],
        a=[[[hx(c), i] for c, i in row] for row in m["a"]],
        b=[[[hx(c), i] for c, i in row] for row in m["b"]],
        alpha_g1=p1(z["alpha_g1"]), beta_g1=p1(z["beta_g1"]), beta_g2=p2(z["beta_g2"]),
        gamma_g2=p2(z["gamma_g2"]), delta_g1=p1(z["delta_g1"]), delta_g2=p2(z["delta_g2"]),
        ic=[p1(P) for P in z["ic"]],
        a_query=[p1(P) for P in z["a_query"]], b_g1_query=[p1(P) for P in z["b_g1_query"]],
        b_g2_query=[p2(P) for P in z["b_g2_query"]], l_query=[p1(P) for P in z["l_query"]],
        h_query=[p1(P) for P in z["h_query"]],
        witness=[hx(x) for x in w], public=[hx(x) for x in pub],
        snarkjs_proof=dict(a=p1(sp[0]), b=p2(sp[1]), c=p1(sp[2])),
        h=[hx(x) for x in h], oracle_proofs=proofs,
    )
    dump("groth16_%s_%s" % (curve_dir, name), obj, compress)


def plonk_fixture(curve_dir, name, expected, compress):
    base = "%s/test_vectors/Plonk/%s/%s/" % (REF, curve_dir, name)
    z = F.read_plonk_zkey(base + "circuit.zkey")
    r, w = F.read_wtns(base + "witness.wtns")
    got = round1_commitments(z, w)
    assert got == expected, "oracle must reproduce the reference KAT"
    # also store the MSM/NTT inputs so the GPU path can be pinned directly on the KAT
    n = z["domain_size"]
    _, roots = roots_of_unity(r)
    gen = roots[n.bit_length() - 1]
    npub = z["n_public"]
    public_inputs = [0] + list(w[1:npub + 1])
    witness = list(w[npub + 1:])
    additions = []

    def get_witness(idx):
        if idx <= npub:
            return public_inputs[idx]
        if idx < z["n_vars"] - z["n_additions"]:
            return witness[idx - npub - 1]
        return additions[idx + z["n_additions"] - z["n_vars"]]

    for s1, s2, f1, f2 in z["additions"]:
        additions.append((get_witness(s1) * f1 + get_witness(s2) * f2) % r)
    wires = []
    blinders = [[0, 1], [2, 3], [4, 5]]
    for wire_map, blind in zip((z["map_a"], z["map_b"], z["map_c"]), blinders):
        buf = [get_witness(i) for i in wire_map] + [0] * (n - len(wire_map))
        poly = ifft(buf, gen, r)
        rev = list(reversed(blind))
        blinded = list(poly)
        for i, c in enumerate(rev):
            blinded[i] = (blinded[i] - c) % r
        blinded += rev
        wires.append(dict(buffer=[hx(x) for x in buf], poly=[hx(x) for x in poly], blinded=[hx(x) for x in blinded]))
    obj = dict(source="test_vectors/Plonk/%s/%s" % (curve_dir, name), curve=curve_dir, domain_size=n,
               group_gen=hx(gen), p_tau=[p1(P) for P in z["p_tau"]], wires=wires,
               expected_commitments=[p1(P) for P in expected],
               expected_source="co-circom/co-plonk/src/round1.rs:351-371" if curve_dir == "bn254" else
               "co-circom/co-plonk/src/round1.rs:397-417")
    dump("plonk_round1_%s_%s" % (curve_dir, name), compact_round1(obj, blinders) if compress else obj, compress)


# The reference's known answers for the whole prover with deterministic blinders b[i] = i on BN254 multiplier2
PLONK_KAT = dict(
    z=((21851995660159341992573113210608672476110709810652234421585224566450425950906,
        9396597540042847815549199092556045933393323370500084953024302516882239981142), "round2.rs:300-306"),
    t1=((14195659590223391588638033663362337117591990036333098666602164584829450067964,
         3556648023705175372561455635244621029434015848660599980046006090530807598362), "round3.rs:611-616"),
    t2=((3735872884021926351213137728148437717828227598563721199864822205706753909354,
         18937554230046023488342718793325695277505320264073327441600348965411357658388), "round3.rs:618-623"),
    t3=((16143856432987537130591639896375147783771732347095191085601174356801897211531,
         181289684093540268434296060454656362990106137005120511426963659280111589561), "round3.rs:625-630"),
    eval_a=(9577617118727487156038114503197927927393325100881782676071854181913228129519, "round4.rs:204-209"),
    eval_b=(20597878711220885145139457487405665380092038394343281979206937623212519986448, "round4.rs:211-216"),
    eval_c=(15265494263612694384441473331344570152140354050926476508657731330784430744915, "round4.rs:218-223"),
    eval_zw=(13208748067365350181326696119359571057028048827339239951085850234164749233153, "round4.rs:225-230"),
    eval_s1=(14333100636430622287126878289812189552775054994479690945797668457655414216377, "round4.rs:232-237"),
    eval_s2=(5227675743165392606371559215386333900775466821923985579976650047914227054429, "round4.rs:239-244"),
    wxi=((17714933343167283383757911844657193439824158284537335005582807825912982308761,
          10956622068891399683012461981563789956666325407769410657364052444385845871778), "round5.rs:394-399"),
    wxiw=((11975595019949715918668172153793336705506375746143971491421022814159658028345,
           21836122222240321064812409945656239690711148338716835775906941056446809090474), "round5.rs:401-406"))
VERIFIER_KAT = dict(  # plonk.rs:266-309, on the snarkjs proof of the same circuit
    alpha=4763880717866883938312853446651867584882243039496717119981221423729366022837,
    beta=21441108096646375017416196030970784867168559532405066373711898693160482621553,
    gamma=18358340056223774859544506185831433076440067236582749990986245668953309272283,
    xi=7090361968641770615455554153830816431169048885260030244909139672173927785729,
    v=[20400998993179279999961662359284658174039203383603729825079844045891169320886,
       14103303087679005329613195828482967369227712227612956336575014332581057266451,
       21001079402417908449694312728019684919907988335857152136145617358865414540686,
       4101776369377085261955299986018358717882425962862873747599549657644387577706,
       2709069871665560223395972486266890200809234039251701259320531117604850964887],
    u=13260637895132000183831258130762201406791497612259050836989270998713858775580)


def plonk_full_fixture(name, compress, curve_dir="bn254", p_tau_from=None):
    """Everything the Plonk prover reads from the zkey (taceo-circom-types plonk::Zkey) + witness, verification
    key, public inputs, the snarkjs proof, and the reference's round 2-5 / verifier known answers."""
    from oracle import plonk as OP
    from oracle.pairing_bn254 import pairing_product_is_one
    base = "%s/test_vectors/Plonk/%s/%s/" % (REF, curve_dir, name)
    z = F.read_plonk_zkey(base + "circuit.zkey")
    _, w = F.read_wtns(base + "witness.wtns")
    vk = F.read_plonk_vk_json(base + "verification_key.json")
    pub = [int(x) for x in json.load(open(base + "public.json"))]
    sp = F.read_plonk_proof_json(base + "circom.proof")
    bn = curve_dir == "bn254"  # the oracle has a pairing for BN254 only
    if bn:
        assert OP.verify(z["curve"], vk, sp, pub, pairing_product_is_one), "snarkjs proof must verify"
    else:
        for k in ("qm", "ql", "qr", "qo", "qc", "s1", "s2", "s3"):
            assert z["vk_" + k] == vk[k], k
    pr = OP.prove(z, w)
    if name == "multiplier2" and bn:
        for k, (val, _) in PLONK_KAT.items():
            assert pr[k] == val, k
        ch = OP.verifier_challenges(z["curve"], vk, sp, pub)
        assert all(ch[k] == v for k, v in VERIFIER_KAT.items())
    if bn:
        assert OP.verify(z["curve"], vk, pr, pub, pairing_product_is_one)
    poly = lambda P: dict(coeffs=[hx(x) for x in P["coeffs"]], evals=[hx(x) for x in P["evals"]])
    pj = lambda P: {k: (p1(v) if isinstance(v, tuple) or v is None else hx(v)) for k, v in P.items()}
    obj = dict(source="test_vectors/Plonk/%s/%s" % (curve_dir, name), curve=curve_dir,
               **{k: z[k] for k in ("n_vars", "n_public", "domain_size", "n_additions", "n_constraints")},
               k1=hx(z["k1"]), k2=hx(z["k2"]), x2=p2(z["x2"]),
               **{"vk_" + k: p1(z["vk_" + k]) for k in ("qm", "ql", "qr", "qo", "qc", "s1", "s2", "s3")},
               additions=[[a, b, hx(c), hx(d)] for a, b, c, d in z["additions"]],
               map_a=z["map_a"], map_b=z["map_b"], map_c=z["map_c"],
               **{k: poly(z[k]) for k in ("qm", "ql", "qr", "qo", "qc", "s1", "s2", "s3")},
               lagrange=[poly(P) for P in z["lagrange"]], p_tau=[p1(P) for P in z["p_tau"]],
               witness=[hx(x) for x in w], public=[hx(x) for x in pub], vk_power=vk["power"],
               snarkjs_proof=pj(sp), oracle_proof_deterministic_blinders=pj(pr),
               oracle_proof_json=F.plonk_proof_to_json(pr, "bn128" if bn else "bls12381"))
    if name == "multiplier2" and bn:
        obj["reference_kat"] = {k: dict(value=(p1(v) if isinstance(v, tuple) else hx(v)), source="co-circom/co-plonk/src/" + src)
                                for k, (v, src) in PLONK_KAT.items()}
        obj["reference_verifier_kat"] = dict(source="co-circom/co-plonk/src/plonk.rs:266-309",
                                             **{k: ([hx(x) for x in v] if isinstance(v, list) else hx(v))
                                                for k, v in VERIFIER_KAT.items()})
    if compress:
        obj = compact_plonk_key(obj, p_tau_from)
    dump("plonk_full_%s_%s" % (curve_dir, name), obj, compress)


def crs_fixture(n):
    pts = F.read_bn254_crs_g1("%s/co-noir/co-noir-common/src/crs/bn254_g1.dat" % REF, n)
    dump("crs_bn254_g1_first%d" % n, dict(source="co-noir/co-noir-common/src/crs/bn254_g1.dat",
                                          points=[p1(P) for P in pts]), True)


def reference_files():
    """The reference's own files that the readers / ingest paths are tested on, under snarkjs/ (zkeys gzipped), and the
    first 64 points of the Ignition CRS file, byte for byte."""
    for rel in ("Groth16/bn254/multiplier2/circuit.zkey", "Groth16/bn254/multiplier2/witness.wtns",
                "Groth16/bn254/poseidon/circuit.zkey", "Groth16/bn254/poseidon/witness.wtns",
                "Groth16/bn254/poseidon/verification_key.json",
                "Groth16/bls12_381/poseidon/circuit.zkey", "Groth16/bls12_381/poseidon/witness.wtns",
                "Groth16/bls12_381/poseidon/verification_key.json", "Groth16/bls12_381/poseidon/circom.proof",
                "Groth16/bls12_381/poseidon/public.json",
                "Plonk/bn254/multiplier2/circuit.zkey", "Plonk/bls12_381/multiplier2/circuit.zkey",
                "Plonk/bls12_381/poseidon/verification_key.json", "Plonk/bls12_381/poseidon/circom.proof",
                "Plonk/bls12_381/poseidon/public.json"):
        data = open("%s/test_vectors/%s" % (REF, rel), "rb").read()
        dst = os.path.join(HERE, "snarkjs", rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        if rel.endswith(".zkey"):
            with gzip.GzipFile(dst + ".gz", "wb", mtime=0) as f:
                f.write(data)
        else:
            open(dst, "wb").write(data)
    crs = open("%s/co-noir/co-noir-common/src/crs/bn254_g1.dat" % REF, "rb").read(64 * 64)
    open(os.path.join(HERE, "crs_bn254_g1_first64.dat"), "wb").write(crs)


if __name__ == "__main__":
    groth16_fixture("multiplier2", [(0, 0), (5, 7)], False)
    groth16_fixture("poseidon", [(123456789, 987654321)], True)
    plonk_fixture("bn254", "multiplier2", [
        (17605081043163307645214588229802469503664729145403357283635330564965670333858,
         6586266374304386912414685272642968153787280144323447197846781700256409557611),
        (5630355441221157622116381279042400483431873694148526624610332736752309357481,
         459435968793897134848228876468434334542717512356212242962101833939899171644),
        (15206827023183180947877311390140741127921188782225553575654415094642569639438,
         14970166502897037710457760872123795383312785044242798403684409588772714154874)], False)
    plonk_fixture("bls12_381", "poseidon", [
        (1998528185362278337803945478659945086542519630073413629642105010067028189206141975508238821825915421715338325238864,
         436066057394619309469331627881449668678557518497178283348448576242129245895320288313540996356612092203769711134939),
        (905523078516729029387874920505888326057985585766807058529621596028494573503715980387105934346404133401227192848784,
         817813208457279034981972137280354075285704598923875006670861630006742541882069169563142367502699866422101983374962),
        (2045702311111033155343546707999313330868835292331631548140598745513449880984849831136790392158415943067742290277175,
         2263708941732971465915801396733005622347769540424301431567098497278413189155761949973582649025461644335372679621757)], True)
    crs_fixture(1024)
    plonk_full_fixture("multiplier2", False)
    plonk_full_fixture("poseidon", True)
    plonk_full_fixture("multiplier2", False, "bls12_381")
    plonk_full_fixture("poseidon", True, "bls12_381", p_tau_from="plonk_round1_bls12_381_poseidon")
    groth16_fixture("multiplier2", [(0, 0), (11, 13)], False, "bls12_381")
    reference_files()
