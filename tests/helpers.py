"""Shared test helpers: golden fixture loading and oracle <-> C-ABI data conversion."""
import gzip
import json
import os

import numpy as np

from co_snarks_b200 import binding as B
from oracle.fields import CURVES, roots_of_unity
from oracle.ntt import fft, ifft

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    p = os.path.join(GOLDEN, name + ".json")
    if os.path.exists(p):
        return json.load(open(p))
    with gzip.open(p + ".gz", "rb") as f:
        g = json.loads(f.read().decode())
    if "sigma" in g:
        _expand_plonk_key(g)
    if "wires" in g and "blinders" in g["wires"][0]:
        _expand_round1(g)
    return g


def _hx(v):
    return format(v, "x")


def _expand_plonk_key(g):
    """Inverse of make_golden.compact_plonk_key: the polynomials in the zkey's layout (n coefficients, then the
    evaluations over the 4n-point domain) from their evaluations over the n-point domain."""
    r, n = CURVES[g["curve"]].r, g["domain_size"]
    _, roots = roots_of_unity(r)
    gen_n, gen_4n = roots[n.bit_length() - 1], roots[n.bit_length() + 1]

    def poly(evals):
        co = ifft(evals, gen_n, r)
        return dict(coeffs=[_hx(x) for x in co], evals=[_hx(x) for x in fft(co + [0] * (3 * n), gen_4n, r)])
    w = [1]
    for _ in range(n - 1):
        w.append(w[-1] * gen_n % r)
    k = (1, ih(g["k1"]), ih(g["k2"]))
    for name, ev in g.pop("q_domain_evals").items():
        g[name] = poly([ih(x) for x in ev])
    for name, sig in zip(("s1", "s2", "s3"), g.pop("sigma")):
        g[name] = poly([k[s // n] * w[s % n] % r for s in sig])
    g["lagrange"] = [poly([int(i == j) for i in range(n)]) for j in range(max(1, g["n_public"]))]
    if "p_tau_from" in g:
        g["p_tau"] = load_golden(g.pop("p_tau_from"))["p_tau"]


def _expand_round1(g):
    """Inverse of make_golden.compact_round1: each wire's polynomial and blinded polynomial."""
    r = CURVES[g["curve"]].r
    for wire in g["wires"]:
        poly = ifft([ih(x) for x in wire["buffer"]], ih(g["group_gen"]), r)
        rev = list(reversed(wire.pop("blinders")))
        blinded = [(c - rev[i]) % r if i < len(rev) else c for i, c in enumerate(poly)] + rev
        wire["poly"], wire["blinded"] = [_hx(x) for x in poly], [_hx(x) for x in blinded]


def golden_fixture(tmp_dir, rel):
    """Path of one of the reference's snarkjs test-vector files kept under golden/snarkjs/<rel>; a file stored
    gzipped is unpacked into tmp_dir first, since the readers under test take a path."""
    p = os.path.join(GOLDEN, "snarkjs", rel)
    if os.path.exists(p):
        return p
    out = os.path.join(str(tmp_dir), rel.replace("/", "_"))
    with gzip.open(p + ".gz", "rb") as f, open(out, "wb") as g:
        g.write(f.read())
    return out


def ih(x):
    return int(x, 16)


def gp1(v):
    return None if v is None else (ih(v[0]), ih(v[1]))


def gp2(v):
    return None if v is None else ((ih(v[0][0]), ih(v[0][1])), (ih(v[1][0]), ih(v[1][1])))


class Conv:
    """Conversions for one curve (oracle ints / tuples <-> Montgomery limb arrays)."""

    def __init__(self, curve_name="bn254"):
        self.c = CURVES[curve_name]
        self.id = B.CS_BN254 if curve_name == "bn254" else B.CS_BLS12_381
        self.q, self.r = self.c.q, self.c.r
        self.nq, self.nr = self.c.nq, 4

    def fr(self, vals):
        vals = list(vals)
        if not vals:
            return np.zeros((0, self.nr), dtype=np.uint64)
        return B.ints_to_limbs(B.to_mont_ints(vals, self.r, self.nr), self.nr)

    def fr_canonical(self, vals):
        return B.ints_to_limbs(list(vals), self.nr)

    def fr_back(self, arr):
        return B.from_mont_ints(B.limbs_to_ints(np.asarray(arr).reshape(-1, self.nr)), self.r, self.nr)

    def g1(self, pts):
        flat = []
        for P in pts:
            flat += [0, 0] if P is None else [P[0], P[1]]
        return B.ints_to_limbs(B.to_mont_ints(flat, self.q, self.nq), self.nq).reshape(len(pts), 2 * self.nq)

    def g2(self, pts):
        flat = []
        for P in pts:
            flat += [0, 0, 0, 0] if P is None else [P[0][0], P[0][1], P[1][0], P[1][1]]
        return B.ints_to_limbs(B.to_mont_ints(flat, self.q, self.nq), self.nq).reshape(len(pts), 4 * self.nq)

    def pt1(self, arr):
        v = B.from_mont_ints(B.limbs_to_ints(np.asarray(arr).reshape(-1, self.nq)), self.q, self.nq)
        return None if not any(v) else (v[0], v[1])

    def pt2(self, arr):
        v = B.from_mont_ints(B.limbs_to_ints(np.asarray(arr).reshape(-1, self.nq)), self.q, self.nq)
        return None if not any(v) else ((v[0], v[1]), (v[2], v[3]))

    def csr(self, rows):
        rp, col, cf = [0], [], []
        for row in rows:
            for c, i in row:
                col.append(i)
                cf.append(c)
            rp.append(len(col))
        return (np.array(rp, dtype=np.uint32), np.array(col, dtype=np.uint32), self.fr(cf))


def golden_groth16(name, curve="bn254"):
    """-> (zkey-like dict, matrices dict, witness ints, golden json) in the oracle's conventions."""
    g = load_golden("groth16_%s_%s" % (curve, name))
    z = dict(curve=CURVES[curve], q=CURVES[curve].q, r=CURVES[curve].r, n_vars=g["n_vars"],
             n_public=g["n_public"], domain_size=g["domain_size"])
    for k in ("alpha_g1", "beta_g1", "delta_g1"):
        z[k] = gp1(g[k])
    for k in ("beta_g2", "gamma_g2", "delta_g2"):
        z[k] = gp2(g[k])
    z["ic"] = [gp1(P) for P in g["ic"]]
    for k in ("a_query", "b_g1_query", "l_query", "h_query"):
        z[k] = [gp1(P) for P in g[k]]
    z["b_g2_query"] = [gp2(P) for P in g["b_g2_query"]]
    m = dict(num_constraints=g["num_constraints"], num_instance_variables=g["num_instance_variables"],
             num_witness_variables=g["num_witness_variables"],
             a=[[(ih(c), i) for c, i in row] for row in g["a"]],
             b=[[(ih(c), i) for c, i in row] for row in g["b"]])
    w = [ih(x) for x in g["witness"]]
    return z, m, w, g


def golden_plonk(name, curve="bn254"):
    """-> (plonk zkey dict in the oracle's conventions, witness ints, golden json)."""
    g = load_golden("plonk_full_%s_%s" % (curve, name))
    c = CURVES[curve]
    z = dict(curve=c, q=c.q, r=c.r)
    for k in ("n_vars", "n_public", "domain_size", "n_additions", "n_constraints", "map_a", "map_b", "map_c"):
        z[k] = g[k]
    z["k1"], z["k2"], z["x2"] = ih(g["k1"]), ih(g["k2"]), gp2(g["x2"])
    poly = lambda P: dict(coeffs=[ih(x) for x in P["coeffs"]], evals=[ih(x) for x in P["evals"]])
    for k in ("qm", "ql", "qr", "qo", "qc", "s1", "s2", "s3"):
        z["vk_" + k] = gp1(g["vk_" + k])
        z[k] = poly(g[k])
    z["lagrange"] = [poly(P) for P in g["lagrange"]]
    z["additions"] = [(a, b, ih(c), ih(d)) for a, b, c, d in g["additions"]]
    z["p_tau"] = [gp1(P) for P in g["p_tau"]]
    return z, [ih(x) for x in g["witness"]], g


def plonk_vk_from_zkey(z, power):
    vk = dict(n_public=z["n_public"], power=power, k1=z["k1"], k2=z["k2"], x2=z["x2"])
    for k in ("qm", "ql", "qr", "qo", "qc", "s1", "s2", "s3"):
        vk[k] = z["vk_" + k]
    return vk


def plonk_proof_from_json(d):
    return {k: (ih(v) if isinstance(v, str) else gp1(v)) for k, v in d.items()}


def plonk_key_arrays(cv, z):
    """oracle-style plonk zkey dict -> the Montgomery limb arrays of cs_plonk_key_desc."""
    na = z["n_additions"]
    return dict(n_vars=z["n_vars"], n_public=z["n_public"], domain_size=z["domain_size"], n_additions=na,
               n_constraints=z["n_constraints"], k1=cv.fr([z["k1"]]), k2=cv.fr([z["k2"]]),
               vk_points=cv.g1([z["vk_" + k] for k in ("qm", "ql", "qr", "qo", "qc", "s1", "s2", "s3")]),
               additions_ids=np.array([[a, b] for a, b, _, _ in z["additions"]], dtype=np.uint32).reshape(na, 2),
               additions_factors=cv.fr([f for _, _, f1, f2 in z["additions"] for f in (f1, f2)]).reshape(na, 2, 4),
               map_a=np.array(z["map_a"], dtype=np.uint32), map_b=np.array(z["map_b"], dtype=np.uint32),
               map_c=np.array(z["map_c"], dtype=np.uint32),
               q_coeffs=[cv.fr(z[k]["coeffs"]) for k in ("qm", "ql", "qr", "qo", "qc")],
               q_evals=[cv.fr(z[k]["evals"]) for k in ("qm", "ql", "qr", "qo", "qc")],
               s_coeffs=[cv.fr(z[k]["coeffs"]) for k in ("s1", "s2", "s3")],
               s_evals=[cv.fr(z[k]["evals"]) for k in ("s1", "s2", "s3")],
               lagrange_evals=np.concatenate([cv.fr(P["evals"]) for P in z["lagrange"]]),
               p_tau=cv.g1(z["p_tau"]))


def make_plonk_key(ctx, cv, z):
    """oracle-style plonk zkey dict -> device PlonkKey."""
    return B.PlonkKey(ctx, cv.id, plonk_key_arrays(cv, z))


def plonk_proof_from_device(cv, pts, evs):
    names = ("a", "b", "c", "z", "t1", "t2", "t3", "wxi", "wxiw")
    proof = {k: cv.pt1(pts[i]) for i, k in enumerate(names)}
    ev = cv.fr_back(evs)
    for i, k in enumerate(("eval_a", "eval_b", "eval_c", "eval_s1", "eval_s2", "eval_zw")):
        proof[k] = ev[i]
    return proof


def make_key(ctx, cv, z, m, window_bits=0):
    mc = dict(num_constraints=m["num_constraints"], num_instance_variables=m["num_instance_variables"],
              num_witness_variables=m["num_witness_variables"], a=cv.csr(m["a"]), b=cv.csr(m["b"]))
    pts = dict(alpha_g1=cv.g1([z["alpha_g1"]]), beta_g1=cv.g1([z["beta_g1"]]), beta_g2=cv.g2([z["beta_g2"]]),
               delta_g1=cv.g1([z["delta_g1"]]), delta_g2=cv.g2([z["delta_g2"]]),
               a_query=cv.g1(z["a_query"]), b_g1_query=cv.g1(z["b_g1_query"]), b_g2_query=cv.g2(z["b_g2_query"]),
               l_query=cv.g1(z["l_query"]), h_query=cv.g1(z["h_query"]))
    return B.Groth16Key(ctx, cv.id, mc, pts, window_bits)
