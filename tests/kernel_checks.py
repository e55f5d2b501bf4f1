"""Parity checks shared by the GPU tests (-m gpu, through libcosnarks_gpu.so) and the CPU-emulation
tests (tests/emu build of the same kernels).  Every check compares the C-ABI result with the oracle
or with a committed golden vector; integer work => bit-exact equality."""
import ctypes as C
import random

import pytest

import numpy as np

from co_snarks_b200 import binding as B
from helpers import GOLDEN, Conv, golden_groth16, gp1, ih, load_golden, make_key
from oracle import groth16 as OG
from oracle import ntt as ON
from oracle.ec import g1 as og1, g2 as og2
from oracle.fields import BN254, CURVES, groth16_roots_of_unity
from oracle.pairing_bn254 import groth16_verify


def check_field_ops(ctx, n=257, seed=1, curve="bn254"):
    cv = Conv(curve)
    r = cv.r
    rng = random.Random(seed)
    a = [rng.randrange(r) for _ in range(n)]
    b = [rng.randrange(r) for _ in range(n)]
    # edge values
    edge = [0, 1, r - 1, r - 2, (r - 1) // 2, 2 ** 253, 2 ** 128 - 1]
    for i, e in enumerate(edge):
        a[i] = e
        b[len(edge) - 1 - i] = e
    da, db = ctx.to_device(cv.fr(a)), ctx.to_device(cv.fr(b))
    do = ctx.alloc(n * 32)
    lib = ctx.lib
    for name, f in (("mul", lambda x, y: x * y % r), ("add", lambda x, y: (x + y) % r), ("sub", lambda x, y: (x - y) % r)):
        ctx._check(getattr(lib, "cs_vec_" + name)(ctx.h, cv.id, da, db, do, n))
        got = cv.fr_back(ctx.d2h(do, (n, 4)))
        assert got == [f(x, y) for x, y in zip(a, b)], "cs_vec_" + name
    # Montgomery conversion helpers and canonical round trip
    can = B.ints_to_limbs(a, 4)
    mont = np.zeros_like(can)
    ctx._check(lib.cs_fr_to_mont(cv.id, B._ptr(can), B._ptr(mont), n))
    assert (mont == cv.fr(a)).all()
    back = np.zeros_like(can)
    ctx._check(lib.cs_fr_from_mont(cv.id, B._ptr(mont), B._ptr(back), n))
    assert (back == can).all()
    for d in (da, db, do):
        ctx.free(d)


def check_share_kernels(ctx, n=300, seed=2):
    cv = Conv("bn254")
    r = cv.r
    rng = random.Random(seed)
    lib = ctx.lib
    a = [(rng.randrange(r), rng.randrange(r)) for _ in range(n)]
    b = [(rng.randrange(r), rng.randrange(r)) for _ in range(n)]
    mask = [rng.randrange(r) for _ in range(n)]
    da = ctx.to_device(cv.fr([x for s in a for x in s]))
    db = ctx.to_device(cv.fr([x for s in b for x in s]))
    dm = ctx.to_device(cv.fr(mask))
    do = ctx.alloc(n * 32)
    ctx._check(lib.cs_rep3_local_mul_vec(ctx.h, cv.id, da, db, dm, do, n))
    assert cv.fr_back(ctx.d2h(do, (n, 4))) == OG.local_mul_vec_rep3(a, b, mask, r)
    ctx._check(lib.cs_rep3_local_mul_vec(ctx.h, cv.id, da, db, None, do, n))
    assert cv.fr_back(ctx.d2h(do, (n, 4))) == OG.local_mul_vec_rep3(a, b, [0] * n, r)
    # distribute_powers on shares (batch 2) and plain (batch 1)
    tab = [rng.randrange(r) for _ in range(n)]
    dt = ctx.to_device(cv.fr(tab))
    ctx._check(lib.cs_vec_scale_table(ctx.h, cv.id, da, dt, n, 2))
    got = cv.fr_back(ctx.d2h(da, (2 * n, 4)))
    assert got == [x * t % r for s, t in zip(a, tab) for x in s]
    ctx._check(lib.cs_vec_scale_table(ctx.h, cv.id, dm, dt, n, 1))
    assert cv.fr_back(ctx.d2h(dm, (n, 4))) == [x * t % r for x, t in zip(mask, tab)]
    # rep3 -> shamir bridge
    ca, cb = rng.randrange(r), rng.randrange(r)
    ctx._check(lib.cs_rep3_to_shamir(ctx.h, cv.id, db, B._ptr(cv.fr([ca])), B._ptr(cv.fr([cb])), do, n))
    assert cv.fr_back(ctx.d2h(do, (n, 4))) == [(ca * x + cb * y) % r for x, y in b]
    for d in (da, db, dm, do, dt):
        ctx.free(d)


def check_roots(ctx):
    cv = Conv("bn254")
    for power in (0, 1, 2, 8, 20, 27, 28):
        gen, shift = ctx.roots_of_unity(cv.id, power)
        eg, es = groth16_roots_of_unity(cv.r, power)
        assert cv.fr_back(gen) == [eg] and cv.fr_back(shift) == [es], power


def check_ntt(ctx, log_sizes, seed=3, curve="bn254"):
    cv = Conv(curve)
    r = cv.r
    rng = random.Random(seed)
    for lg in log_sizes:
        n = 1 << lg
        g, _ = groth16_roots_of_unity(r, lg)
        dom = ctx.domain(cv.id, lg, cv.fr([g]))
        assert dom.size() == n
        for batch in (1, 2):
            v = [rng.randrange(r) for _ in range(n * batch)]
            arr = cv.fr(v)
            dom.ifft_in_to_out(arr, batch)
            exp = [None] * (n * batch)
            for c in range(batch):
                exp[c::batch] = ON.ifft_in_to_out(v[c::batch], g, r)
            assert cv.fr_back(arr) == exp, ("ifft_in_to_out", lg, batch)
            dom.fft_out_to_in(arr, batch)
            assert cv.fr_back(arr) == v, ("fft_out_to_in", lg, batch)
        # bit_reverse
        v = [rng.randrange(r) for _ in range(n)]
        d = ctx.to_device(cv.fr(v))
        ctx._check(ctx.lib.cs_bit_reverse(ctx.h, cv.id, d, lg, 1))
        assert cv.fr_back(ctx.d2h(d, (n, 4))) == ON.bit_reverse_perm(v)
        ctx.free(d)
        dom.free()


def _edge_case_inputs(G, gen, n, r, rng):
    pts = [G.mul(gen, rng.randrange(1, r)) for _ in range(n)]
    sc = [rng.randrange(r) for _ in range(n)]
    if n >= 12:
        pts[5] = None           # infinity base
        pts[7] = pts[6]         # duplicate base, equal scalars -> P + P inside a bucket
        pts[9] = G.neg(pts[8])  # negated base, equal scalars -> P + (-P)
        sc[0], sc[1], sc[2] = 0, 1, r - 1
        sc[6] = sc[7] = 12345
        sc[8] = sc[9] = 777
    return pts, sc


def check_msm(ctx, group, n, window_bits=(0,), seed=4, curve="bn254"):
    cv = Conv(curve)
    r = cv.r
    rng = random.Random(seed + group)
    C = CURVES[curve]
    G = og1(C) if group == 0 else og2(C)
    gen = C.g1 if group == 0 else C.g2
    to_arr = cv.g1 if group == 0 else cv.g2
    to_pt = cv.pt1 if group == 0 else cv.pt2
    pts, sc = _edge_case_inputs(G, gen, n, r, rng)
    exp = G.msm(pts, sc)
    for wb in window_bits:
        bases = ctx.bases_upload(cv.id, group, to_arr(pts), wb)
        assert len(bases) == n
        out, inf = ctx.msm(bases, cv.fr(sc), montgomery=True)      # msm_unchecked(&[Fr])
        assert to_pt(out) == exp and inf == (exp is None), ("msm mont", group, wb)
        out, inf = ctx.msm(bases, cv.fr_canonical(sc), montgomery=False)  # msm_bigint
        assert to_pt(out) == exp, ("msm bigint", group, wb)
        # sub-slice (query[1 + pub ..]) and ragged n
        for off, cnt in ((1, n - 1), (3, 1), (n // 3, n // 2)):
            out, inf = ctx.msm(bases, cv.fr(sc[off:off + cnt]), offset=off)
            assert to_pt(out) == G.msm(pts[off:off + cnt], sc[off:off + cnt]), ("slice", off, cnt)
        # empty input -> identity
        out, inf = ctx.msm(bases, np.zeros((0, 4), dtype=np.uint64))
        assert inf and to_pt(out) is None
        # all-zero scalars -> identity
        out, inf = ctx.msm(bases, cv.fr([0] * n))
        assert inf and to_pt(out) is None
        # heavy skew: every scalar equal (one bucket per window takes all points)
        out, inf = ctx.msm(bases, cv.fr([3] * n))
        assert to_pt(out) == G.msm(pts, [3] * n)
        if n >= 12:
            out, inf = ctx.msm(bases, cv.fr([5, 5]), offset=8)  # P + (-P)
            assert inf
        bases.free()


def check_msm_crs(ctx):
    """MSM over real Ignition CRS points (co-noir-common/src/crs/bn254_g1.dat, first 1024)."""
    cv = Conv("bn254")
    g = load_golden("crs_bn254_g1_first1024")
    pts = [gp1(P) for P in g["points"]]
    assert pts[0] == (1, 2)
    rng = random.Random(11)
    sc = [rng.randrange(cv.r) for _ in pts]
    bases = ctx.bases_upload(cv.id, 0, cv.g1(pts))
    out, _ = ctx.msm(bases, cv.fr(sc))
    assert cv.pt1(out) == og1(BN254).msm(pts, sc)
    bases.free()


def check_crs_file_ingest(ctx, tmp_path):
    """cs_bases_from_crs_file on a file in the bn254_g1.dat layout (64 B/point, big-endian canonical;
    co-noir-common/src/crs/parse.rs:93-101) written from the golden Ignition points: MSM == oracle, with an offset."""
    import os
    cv = Conv("bn254")
    g = load_golden("crs_bn254_g1_first1024")
    pts = [gp1(P) for P in g["points"]][:300]
    path = os.path.join(str(tmp_path), "g1.dat")
    with open(path, "wb") as f:
        for x, y in pts:
            f.write(x.to_bytes(32, "big") + y.to_bytes(32, "big"))
    rng = random.Random(12)
    for off, n in ((0, 300), (7, 200)):
        bases = ctx.bases_from_crs_file(path, n, off)
        sc = [rng.randrange(cv.r) for _ in range(n)]
        out, _ = ctx.msm(bases, cv.fr(sc))
        assert cv.pt1(out) == og1(BN254).msm(pts[off:off + n], sc)
        bases.free()
    with pytest.raises(RuntimeError):
        ctx.bases_from_crs_file(path, 400)  # more points than the file holds
    # the first 64 points of the real file, byte for byte: its first point is the generator
    bases = ctx.bases_from_crs_file(os.path.join(GOLDEN, "crs_bn254_g1_first64.dat"), 64)
    out, _ = ctx.msm(bases, cv.fr([1] + [0] * 63))
    assert cv.pt1(out) == (1, 2)
    bases.free()


def check_fixed_base_mul(ctx, n=40):
    cv = Conv("bn254")
    rng = random.Random(6)
    sc = [rng.randrange(cv.r) for _ in range(n)]
    sc[0], sc[1] = 0, 1
    for group, G, gen, to_arr, to_pt in ((0, og1(BN254), BN254.g1, cv.g1, cv.pt1), (1, og2(BN254), BN254.g2, cv.g2, cv.pt2)):
        out = ctx.fixed_base_mul(cv.id, group, to_arr([gen])[0], cv.fr(sc))
        assert [to_pt(o) for o in out] == [G.mul(gen, s) for s in sc]


def check_plonk_round1_kat(ctx, curve="bn254", name="multiplier2"):
    """GPU iNTT + MSM against the REFERENCE'S known answers (co-plonk/src/round1.rs:351-371)."""
    g = load_golden("plonk_round1_%s_%s" % (curve, name))
    cv = Conv(curve)
    n = g["domain_size"]
    lg = n.bit_length() - 1
    gen = ih(g["group_gen"])
    dom = ctx.domain(cv.id, lg, cv.fr([gen]))
    p_tau = [gp1(P) for P in g["p_tau"]]
    bases = ctx.bases_upload(cv.id, 0, cv.g1(p_tau))
    for wire, exp in zip(g["wires"], g["expected_commitments"]):
        buf = [ih(x) for x in wire["buffer"]]
        # ifft (natural -> natural) = ifft_in_to_out followed by bit_reverse
        d = ctx.to_device(cv.fr(buf))
        dom.ifft_in_to_out(d, 1)
        ctx._check(ctx.lib.cs_bit_reverse(ctx.h, cv.id, d, lg, 1))
        poly = cv.fr_back(ctx.d2h(d, (n, 4)))
        ctx.free(d)
        assert poly == [ih(x) for x in wire["poly"]]
        blinded = [ih(x) for x in wire["blinded"]]
        out, _ = ctx.msm(bases, cv.fr(blinded), n=len(blinded))
        assert cv.pt1(out) == gp1(exp), "commitment differs from the reference KAT"
    bases.free()
    dom.free()


def check_groth16_fixture(ctx, name, rep3=True, window_bits=0, curve="bn254"):
    cv = Conv(curve)
    r = cv.r
    z, m, w, g = golden_groth16(name, curve)
    verify = groth16_verify
    if curve == "bls12_381":
        from oracle.pairing_bls12_381 import groth16_verify as verify
    ni = m["num_instance_variables"]
    pk = make_key(ctx, cv, z, m, window_bits)
    assert pk.domain_size() == g["domain_size"]
    pub, wit = cv.fr(w[:ni]), cv.fr(w[ni:])
    h_exp = [ih(x) for x in g["h"]]
    assert cv.fr_back(pk.witness_map(pub, wit)) == h_exp, "witness map"
    vk = OG.vk_from_zkey(z)
    public = [ih(x) for x in g["public"]]
    for pr in g["oracle_proofs"]:
        A, Bp, Cp = pk.prove_plain(pub, wit, cv.fr([ih(pr["r"])]), cv.fr([ih(pr["s"])]))
        proof = (cv.pt1(A), cv.pt2(Bp), cv.pt1(Cp))
        from oracle.formats import proof_to_json
        assert proof_to_json(*proof, "bn128" if curve == "bn254" else "bls12381") == pr["json"], \
            "proof bytes differ from the oracle for fixed (r, s)"
        assert verify(vk, public, proof)
    if rep3:
        check_groth16_rep3_local(ctx, pk, cv, z, m, w, h_exp, vk, public)
    pk.free()


def check_groth16_rep3_local(ctx, pk, cv, z, m, w, h_exp, vk, public, seed=5):
    """Three parties' local phases on one context, then the reference's two network legs emulated in
    the test (groth16.rs:296-337): the opened proof must equal the plain proof for r = sum r_i.a."""
    r = cv.r
    rng = random.Random(seed)
    ni = m["num_instance_variables"]
    n = pk.domain_size()
    lib = ctx.lib
    wsh = OG.share_rep3(w[ni:], r, rng)

    def zero_masks(k):
        prf = [[rng.randrange(r) for _ in range(k)] for _ in range(3)]
        return [[(prf[i][j] - prf[(i + 2) % 3][j]) % r for j in range(k)] for i in range(3)]

    m1, m2 = zero_masks(n), zero_masks(n)
    rsh = OG.share_rep3([rng.randrange(r)], r, rng)
    ssh = OG.share_rep3([rng.randrange(r)], r, rng)
    rs_mask = zero_masks(1)
    pub = cv.fr(w[:ni])
    loc = []
    h_tot = [0] * n
    for i in range(3):
        sh = cv.fr([x for ab in wsh[i] for x in ab])
        hh = pk.witness_map(pub, sh, B.CS_REP3, i, cv.fr(m1[i]), cv.fr(m2[i]))
        h_i = cv.fr_back(hh)
        assert h_i == OG.witness_map_rep3(i, m, w[:ni], wsh[i], m1[i], m2[i], r, 28)
        h_tot = [(x + y) % r for x, y in zip(h_tot, h_i)]
        loc.append(pk.rep3_local(i, pub, sh, cv.fr(m1[i]), cv.fr(m2[i]), cv.fr(list(rsh[i][0])), cv.fr(list(ssh[i][0]))))
    assert h_tot == h_exp
    G1, G2 = og1(BN254), og2(BN254)
    # open_half_point(A)
    A = None
    for i in range(3):
        A = G1.add(A, cv.pt1(loc[i][0]))
    gC = []
    for i in range(3):
        pa, pb = cv.pt1(loc[i][1]), cv.pt1(loc[(i + 2) % 3][1])
        ra, rb = rsh[i][0]
        r_b1 = G1.add(G1.add(G1.mul(pa, ra), G1.mul(pa, rb)), G1.mul(pb, ra))  # EC masks omitted: they cancel
        rs_i = OG.local_mul_vec_rep3([rsh[i][0]], [ssh[i][0]], [rs_mask[i][0]], r)[0]
        c = G1.add(G1.mul(A, ssh[i][0][0]), r_b1)
        c = G1.add(c, G1.neg(G1.mul(z["delta_g1"], rs_i)))
        c = G1.add(G1.add(c, cv.pt1(loc[i][3])), cv.pt1(loc[i][4]))
        gC.append(c)
    C, Bp = None, None
    for i in range(3):
        C = G1.add(C, gC[i])
        Bp = G2.add(Bp, cv.pt2(loc[i][2]))
    r_tot = sum(x[0][0] for x in rsh) % r
    s_tot = sum(x[0][0] for x in ssh) % r
    assert (A, Bp, C) == OG.prove_plain(z, m, w, r_tot, s_tot)
    assert groth16_verify(vk, public, (A, Bp, C))


def check_msm_rep3_shares(ctx, n=200, seed=8):
    """rep3::pointshare::msm_public_points: both share components from the interleaved array."""
    cv = Conv("bn254")
    rng = random.Random(seed)
    G = og1(BN254)
    pts = [G.mul(BN254.g1, rng.randrange(1, cv.r)) for _ in range(n)]
    sh = [(rng.randrange(cv.r), rng.randrange(cv.r)) for _ in range(n)]
    bases = ctx.bases_upload(cv.id, 0, cv.g1(pts))
    oa, ob = ctx.msm_rep3_shares(bases, cv.fr([x for s in sh for x in s]).reshape(n, 8))
    assert cv.pt1(oa) == G.msm(pts, [s[0] for s in sh]) and cv.pt1(ob) == G.msm(pts, [s[1] for s in sh])
    bases.free()


def check_groth16_shamir_local(ctx, name="multiplier2", seed=9):
    """ShamirCoGroth16 (t = 1, n = 3, the only valid 3-party setting: shamir.rs:41-43): the three
    parties' local phases on degree-1 shares, opened by Lagrange interpolation at 0 with weights
    (3, -3, 1) as degree-2 sharings (shamir/pointshare.rs:102-111), give the plain proof for
    r = r(0), s = s(0)."""
    cv = Conv("bn254")
    r = cv.r
    rng = random.Random(seed)
    z, m, w, g = golden_groth16(name)
    ni = m["num_instance_variables"]
    pk = make_key(ctx, cv, z, m)
    G1, G2 = og1(BN254), og2(BN254)

    def shamir(v):  # degree-1 polynomial, party i evaluates at i + 1
        a = rng.randrange(r)
        return [(v + a * (i + 1)) % r for i in range(3)]

    wsh = [shamir(x) for x in w[ni:]]
    r0, s0 = rng.randrange(r), rng.randrange(r)
    rsh, ssh = shamir(r0), shamir(s0)
    lam = [3, r - 3, 1]
    pub = cv.fr(w[:ni])
    loc = [pk.shamir_local(pub, cv.fr([x[i] for x in wsh]), cv.fr([rsh[i]]), cv.fr([ssh[i]])) for i in range(3)]

    def open_(pts, G):
        acc = None
        for P, l in zip(pts, lam):
            acc = G.add(acc, G.mul(P, l))
        return acc

    A = open_([cv.pt1(loc[i][0]) for i in range(3)], G1)
    Bp = open_([cv.pt2(loc[i][2]) for i in range(3)], G2)
    gc = []
    for i in range(3):
        c = G1.add(G1.mul(A, ssh[i]), G1.mul(cv.pt1(loc[i][1]), rsh[i]))
        c = G1.add(c, G1.neg(G1.mul(z["delta_g1"], rsh[i] * ssh[i] % r)))
        c = G1.add(G1.add(c, cv.pt1(loc[i][3])), cv.pt1(loc[i][4]))
        gc.append(c)
    C = open_(gc, G1)
    assert (A, Bp, C) == OG.prove_plain(z, m, w, r0, s0)
    pk.free()


def check_plonk_primitives(ctx, lg=9, seed=10):
    """co-plonk building blocks: natural-order fft/ifft on the n and 4n domains (types.rs:76-100) and
    evaluate_poly_public / eval_poly on shares (rep3/poly.rs:42-68)."""
    from oracle.fields import roots_of_unity
    cv = Conv("bn254")
    r = cv.r
    rng = random.Random(seed)
    _, roots = roots_of_unity(r)
    n = 1 << lg
    for size_lg in (lg, lg + 2):
        N = 1 << size_lg
        g = roots[size_lg]
        dom = ctx.domain(cv.id, size_lg, cv.fr([g]))
        for batch in (1, 2):
            v = [rng.randrange(r) for _ in range(n * batch)] + [0] * ((N - n) * batch)  # zero-padded like arkworks
            d = ctx.to_device(cv.fr(v))
            dom.fft(d, batch)
            got = cv.fr_back(ctx.d2h(d, (N * batch, 4)))
            exp = [None] * (N * batch)
            for c in range(batch):
                exp[c::batch] = ON.fft(v[c::batch], g, r)
            assert got == exp, ("fft", size_lg, batch)
            dom.ifft(d, batch)
            assert cv.fr_back(ctx.d2h(d, (N * batch, 4))) == v, ("ifft", size_lg, batch)
            ctx.free(d)
        dom.free()
    # polynomial evaluation at a public point, plain and shared, ragged length
    for ncoef in (1, 63, 64, 65, 1000, 8192 + 5):
        for batch in (1, 2):
            co = [rng.randrange(r) for _ in range(ncoef * batch)]
            x = rng.randrange(r)
            d = ctx.to_device(cv.fr(co))
            got = cv.fr_back(ctx.eval_poly(cv.id, d, ncoef, cv.fr([x])[0], batch))
            exp = []
            for c in range(batch):
                acc = 0
                for k in reversed(co[c::batch]):
                    acc = (acc * x + k) % r
                exp.append(acc)
            assert got == exp, ("eval_poly", ncoef, batch)
            ctx.free(d)
    # point = 0 -> constant term (poly.rs:43-45)
    d = ctx.to_device(cv.fr([7, 8, 9]))
    assert cv.fr_back(ctx.eval_poly(cv.id, d, 3, cv.fr([0])[0], 1)) == [7]
    ctx.free(d)


def check_rep3_mask_prf(ctx, n=100):
    """On-device ChaCha PRF: block function == RFC 7539 2.3.2 (20 rounds), 12-round keystream and the
    mask vector == the oracle's restatement of Rep3Rand::masking_field_elements_vec (rngs.rs:137-156),
    and the three parties' masks cancel (rngs.rs:103-106)."""
    import struct
    from oracle import chacha as OC
    cv = Conv("bn254")
    key = bytes(range(32))
    # RFC 7539 section 2.3.2: counter = 1, nonce 00000009 0000004a 00000000 -> expressed through the 64-bit
    # counter's high word; the stream-id words are fixed to 0 on the device, so compare via the oracle.
    ks = ctx.chacha_keystream(key, 5, 12, 3)
    assert list(ks) == OC.keystream_words(key, 5 * 16, 48, 12)
    ks20 = ctx.chacha_keystream(key, 1, 20, 1)
    assert list(ks20) == OC.block(struct.unpack("<8I", key), 1, 0, 20)
    # published known answer (draft-strombergson-chacha-test-vectors-01, TC1, 12 rounds: zero key, block 0)
    assert bytes(np.asarray(ctx.chacha_keystream(bytes(32), 0, 12, 1), dtype="<u4").tobytes()).hex().startswith(
        "9bf49a6a0755f953811fce125f2683d50429c3bb49e074147e0089a52eae155f")
    seeds = [bytes((7 * p + i) & 0xff for i in range(32)) for p in range(3)]
    pos = [16, 3, 40]  # word positions, deliberately not block-aligned
    tot = [0] * n
    for p in range(3):
        prev = (p + 2) % 3
        d = ctx.alloc(n * 32)
        ctx.rep3_masks_device(cv.id, seeds[p], pos[p], seeds[prev], pos[prev], n, d)
        got = cv.fr_back(ctx.d2h(d, (n, 4)))
        ctx.free(d)
        assert got == OC.masking_field_elements_vec(seeds[p], pos[p], seeds[prev], pos[prev], n, cv.r)
        tot = [(x + y) % cv.r for x, y in zip(tot, got)]
    assert tot == [0] * n


def check_rep3_mul_vec_reshare(ctx, n=150, seed=15, use_ipc=False):
    """mul_vec as one kernel (local_mul_vec + reshare_vec, arithmetic.rs:132-160): three parties in one
    address space, each storing its z into its own .a and -- through an IPC-mapped pointer -- into the next
    party's .b.  Checks: z == oracle (share product + ChaCha masks), shares are consistent (b of party i ==
    a of party i-1) and open to x*y; the staging variant (cs_rep3_set_b) gives the same vectors."""
    from oracle import chacha as OC
    cv = Conv("bn254")
    r = cv.r
    rng = random.Random(seed)
    xs = [rng.randrange(r) for _ in range(n)]
    ys = [rng.randrange(r) for _ in range(n)]

    def share(v):
        s0, s1 = rng.randrange(r), rng.randrange(r)
        sh = [s0, s1, (v - s0 - s1) % r]
        return [(sh[p], sh[(p + 2) % 3]) for p in range(3)]  # party p holds (x_p, x_{p-1})  rep3.rs:281-293
    xsh = [share(v) for v in xs]
    ysh = [share(v) for v in ys]
    seeds = [bytes((11 * p + i) & 0xff for i in range(32)) for p in range(3)]
    pos = [0, 24, 7]
    d_a, d_b, d_out, d_out2 = [], [], [], []
    for p in range(3):
        d_a.append(ctx.to_device(cv.fr([c for i in range(n) for c in xsh[i][p]])))
        d_b.append(ctx.to_device(cv.fr([c for i in range(n) for c in ysh[i][p]])))
        d_out.append(ctx.alloc(n * 64))
        d_out2.append(ctx.alloc(n * 64))
    # a CUDA IPC handle cannot be opened by the process that exported it: one-process runs on a real GPU pass
    # the neighbour's pointer directly; the IPC mapping itself is exercised by tests/test_dist_rep3.py on GPUs
    peers = [ctx.ipc_open(ctx.ipc_export(d_out[(p + 1) % 3])) if use_ipc else d_out[(p + 1) % 3] for p in range(3)]
    for p in range(3):
        prev = (p + 2) % 3
        ctx.rep3_mul_vec_reshare(cv.id, d_a[p], d_b[p], n, (seeds[p], pos[p], seeds[prev], pos[prev], 12), d_out[p], peers[p])
    ctx.synchronize()
    got = [cv.fr_back(ctx.d2h(d_out[p], (2 * n, 4))) for p in range(3)]
    for p in range(3):
        prev = (p + 2) % 3
        masks = OC.masking_field_elements_vec(seeds[p], pos[p], seeds[prev], pos[prev], n, r)
        exp = [(xsh[i][p][0] * ysh[i][p][0] + xsh[i][p][0] * ysh[i][p][1] + xsh[i][p][1] * ysh[i][p][0] + masks[i]) % r
               for i in range(n)]
        assert got[p][0::2] == exp, ("z", p)
        assert got[p][1::2] == got[prev][0::2], ("reshare", p)
    assert [(got[0][2 * i] + got[1][2 * i] + got[2][2 * i]) % r for i in range(n)] == [x * y % r for x, y in zip(xs, ys)]
    # staging-buffer variant: same z without a peer pointer, b-halves delivered as contiguous vectors
    for p in range(3):
        prev = (p + 2) % 3
        ctx.rep3_mul_vec_reshare(cv.id, d_a[p], d_b[p], n, (seeds[p], pos[p], seeds[prev], pos[prev], 12), d_out2[p], None)
    ctx.synchronize()
    for p in range(3):
        prev = (p + 2) % 3
        zprev = ctx.d2h(d_out2[prev], (2 * n, 4))[0::2].copy()
        d_recv = ctx.to_device(zprev)
        ctx.rep3_set_b(cv.id, d_recv, n, d_out2[p])
        ctx.synchronize()
        ctx.free(d_recv)
    for p in range(3):
        assert cv.fr_back(ctx.d2h(d_out2[p], (2 * n, 4))) == got[p], ("staging", p)
    # no masks (prf NULL) -> plain share product
    ctx.rep3_mul_vec_reshare(cv.id, d_a[0], d_b[0], n, None, d_out2[0], None)
    ctx.synchronize()
    z0 = cv.fr_back(ctx.d2h(d_out2[0], (2 * n, 4)))[0::2]
    assert z0 == [(xsh[i][0][0] * (ysh[i][0][0] + ysh[i][0][1]) + xsh[i][0][1] * ysh[i][0][0]) % r for i in range(n)]
    for p in range(3):
        if use_ipc:
            ctx.ipc_close(peers[p])
        for d in (d_a[p], d_b[p], d_out[p], d_out2[p]):
            ctx.free(d)


def check_keccak(lib):
    from oracle import plonk as OP
    for msg in (b"", b"abc", bytes(range(135)), bytes(range(136)), bytes(200) + b"x" * 77):
        assert B.keccak256(lib, msg) == OP.keccak256(msg)
    assert B.keccak256(lib, b"").hex() == "c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470"


def check_plonk_prove(ctx, name="multiplier2", random_blinders=True, curve="bn254"):
    """Plonk::plain_prove on the device == the oracle's restatement, field by field, for the reference's
    deterministic blinders (the KAT setting of co-plonk/src/round{2..5}.rs tests) and for random ones; the proof
    JSON equals the committed golden one, which the oracle's verifier accepts (tests/test_oracle_golden.py)."""
    from helpers import golden_plonk, make_plonk_key, plonk_proof_from_device
    from oracle import plonk as OP
    from oracle.formats import plonk_proof_to_json
    cv = Conv(curve)
    z, w, g = golden_plonk(name, curve)
    npub = z["n_public"]
    pk = make_plonk_key(ctx, cv, z)
    pub, wit = cv.fr(w[:npub + 1]), cv.fr(w[npub + 1:])
    pts, evs = pk.prove_plain(pub, wit, cv.fr(list(range(11))))
    got = plonk_proof_from_device(cv, pts, evs)
    assert plonk_proof_to_json(got, g["oracle_proof_json"]["curve"]) == g["oracle_proof_json"]
    if "reference_kat" in g:
        for k, kat in g["reference_kat"].items():
            exp = gp1(kat["value"]) if isinstance(kat["value"], list) else ih(kat["value"])
            assert got[k] == exp, (k, kat["source"])
    if random_blinders:
        rng = random.Random(17)
        bl = [rng.randrange(cv.r) for _ in range(11)]
        pts, evs = pk.prove_plain(pub, wit, cv.fr(bl))
        assert plonk_proof_from_device(cv, pts, evs) == OP.prove(z, w, bl)
    # error behaviour: wrong witness length (PlonkProofError::CorruptedWitness territory, lib.rs:60-62)
    with pytest.raises(RuntimeError):
        pk.prove_plain(pub, wit[:-1], cv.fr(list(range(11))))
    pk.free()


def check_plonk_zkey_ingest(ctx, tmp_path, name="multiplier2", curve="bn254"):
    """cs_plonk_pk_from_zkey: a snarkjs-format Plonk .zkey written from the golden fixture, and the reference's own
    file, go straight to the device layout; the proof equals the golden one."""
    import os
    from helpers import golden_fixture, golden_plonk, plonk_proof_from_device
    from oracle import formats as F
    from zkey_writer import write_plonk_zkey
    cv = Conv(curve)
    z, w, g = golden_plonk(name, curve)
    path = os.path.join(str(tmp_path), "plonk_%s_%s.zkey" % (curve, name))
    write_plonk_zkey(path, z)
    back = F.read_plonk_zkey(path)
    assert all(back[k] == z[k] for k in ("k1", "k2", "map_a", "additions", "qm", "s3", "lagrange", "p_tau", "x2", "vk_s2"))
    paths = [path, golden_fixture(tmp_path, "Plonk/%s/%s/circuit.zkey" % (curve, name))]
    npub = z["n_public"]
    for pth in paths:
        pk = B.PlonkKey.from_zkey(ctx, pth, cv.id)
        assert pk.n_public == npub and pk.n_witness == len(w) - npub - 1
        pts, evs = pk.prove_plain(cv.fr(w[:npub + 1]), cv.fr(w[npub + 1:]), cv.fr(list(range(11))))
        got = plonk_proof_from_device(cv, pts, evs)
        assert F.plonk_proof_to_json(got, g["oracle_proof_json"]["curve"]) == g["oracle_proof_json"], pth
        pk.free()
    with pytest.raises(RuntimeError):
        B.PlonkKey.from_zkey(ctx, os.path.join(str(tmp_path), "missing.zkey"), cv.id)


def check_plonk_key_errors(ctx):
    """PlonkProofError behaviour at the boundary (co-plonk/src/lib.rs:40-69, types.rs:79-84): invalid domain size,
    SRS too short for the blinded polynomials, wire maps / additions that index past the witness."""
    import copy
    from helpers import golden_plonk, make_plonk_key
    cv = Conv("bn254")
    z, w, g = golden_plonk("multiplier2")

    def expect(mut, text):
        z2 = copy.deepcopy({k: v for k, v in z.items() if k != "curve"})
        z2["curve"] = z["curve"]
        mut(z2)
        with pytest.raises(RuntimeError) as e:
            make_plonk_key(ctx, cv, z2).free()
        assert text in str(e.value), str(e.value)

    def bad_domain(z2):
        z2["domain_size"] = 6
    expect(bad_domain, "Invalid domain size")

    def short_srs(z2):
        z2["p_tau"] = z2["p_tau"][:z2["domain_size"] + 5]
    expect(short_srs, "SRS points")

    def bad_map(z2):
        z2["map_b"] = list(z2["map_b"])
        z2["map_b"][0] = z2["n_vars"]
    expect(bad_map, "Cannot index into witness")
    # a well-formed key still loads afterwards
    make_plonk_key(ctx, cv, z).free()


def check_plonk_synthetic(ctx, log_n, n_public=2, against_oracle=True, seed=5):
    """Synthetic snarkjs-style key with known tau (workloads/synth_plonk.py): the device proof is accepted by the
    oracle's verifier (pairing check) and rejected for a wrong public input; at small sizes it also equals the
    oracle prover's proof bit for bit.  Covers additions with dependency levels, empty rows and n_public = 0."""
    from helpers import plonk_proof_from_device
    from oracle import plonk as OP
    from oracle.pairing_bn254 import pairing_product_is_one
    from workloads.synth_plonk import SynthPlonk
    cv = Conv("bn254")
    syn = SynthPlonk(ctx, log_n, n_public=n_public)
    pk = syn.make_key()
    rng = random.Random(seed)
    bl = [rng.randrange(cv.r) for _ in range(11)]
    pts, evs = pk.prove_plain(syn.public_inputs, syn.private_witness, cv.fr(bl))
    got = plonk_proof_from_device(cv, pts, evs)
    pub = syn.full_witness[1:n_public + 1]
    vk = syn.vk_ints()
    assert OP.verify(BN254, vk, got, pub, pairing_product_is_one)
    if n_public:
        assert not OP.verify(BN254, vk, got, [(pub[0] + 1) % cv.r] + pub[1:], pairing_product_is_one)
    if against_oracle:
        assert OP.prove(syn.oracle_zkey(), syn.full_witness, bl) == got
    pk.free()


def _plonk_rep3_in_process(ctx, cv, pk, z_n, vk_points, pub, w_private, blinders, seed=23, draw_blinders=False):
    """Three Rep3 co-Plonk parties in one process (LocalRep3Comm) on shares of `w_private` and of `blinders`."""
    from co_snarks_b200.plonk import LocalRep3Comm, Rep3CoPlonk
    from co_snarks_b200.rep3 import Rep3State
    rng = random.Random(seed)
    r = cv.r

    def share(vals):
        out = [[], [], []]
        for v in vals:
            s0, s1 = rng.randrange(r), rng.randrange(r)
            sh = [s0, s1, (v - s0 - s1) % r]
            for p in range(3):
                out[p] += [sh[p], sh[(p + 2) % 3]]  # party p holds (x_p, x_{p-1})  rep3.rs:281-293
        return [cv.fr(o).reshape(-1, 2, 4) for o in out]
    wsh = share(w_private)
    bsh = [None] * 3 if draw_blinders else share(blinders)  # None: Round1Challenges::random via T::rand (round1.rs:82-92)
    seeds = [bytes((31 * p + i) & 0xff for i in range(32)) for p in range(3)]
    provers = [Rep3CoPlonk(ctx, pk, p) for p in range(3)]
    states = [Rep3State.from_seeds(p, seeds[p], seeds[(p + 2) % 3]) for p in range(3)]
    comm = LocalRep3Comm(provers)
    res = comm.run([provers[p].prove(states[p], pub, wsh[p], vk_points, z_n, bsh[p]) for p in range(3)])
    for p in provers:
        p.free()
    # consistent PRF consumption (party p's stream 1 is party p+1's stream 2)
    assert all(states[p].rng1.pos == states[(p + 1) % 3].rng2.pos for p in range(3))
    return res


def check_plonk_rep3(ctx, name="multiplier2"):
    """Rep3CoPlonk::prove (co-plonk/src/lib.rs:222-240) with three parties: every party opens the same proof, and
    it equals the plain prover's (= the oracle's, = the reference's known answers for b = [0..11)) because the
    blinder shares sum to b and all masks cancel."""
    from helpers import golden_plonk, make_plonk_key, plonk_proof_from_device
    from oracle.formats import plonk_proof_to_json
    cv = Conv("bn254")
    z, w, g = golden_plonk(name)
    npub = z["n_public"]
    pk = make_plonk_key(ctx, cv, z)
    vkp = cv.g1([z["vk_" + k] for k in ("qm", "ql", "qr", "qo", "qc", "s1", "s2", "s3")])
    res = _plonk_rep3_in_process(ctx, cv, pk, z["domain_size"], vkp, cv.fr(w[:npub + 1]), w[npub + 1:], list(range(11)))
    proofs = [plonk_proof_from_device(cv, pts, evs) for pts, evs in res]
    assert proofs[0] == proofs[1] == proofs[2]
    assert plonk_proof_to_json(proofs[0]) == g["oracle_proof_json"]
    pk.free()


def check_plonk_rep3_drawn_blinders(ctx, name="multiplier2"):
    """The production path: each party draws its blinder shares from its correlated streams (arithmetic::rand).
    All parties open the same proof and Plonk::verify accepts it."""
    from helpers import golden_plonk, make_plonk_key, plonk_proof_from_device, plonk_vk_from_zkey
    from oracle import plonk as OP
    from oracle.pairing_bn254 import pairing_product_is_one
    cv = Conv("bn254")
    z, w, g = golden_plonk(name)
    npub = z["n_public"]
    pk = make_plonk_key(ctx, cv, z)
    vkp = cv.g1([z["vk_" + k] for k in ("qm", "ql", "qr", "qo", "qc", "s1", "s2", "s3")])
    res = _plonk_rep3_in_process(ctx, cv, pk, z["domain_size"], vkp, cv.fr(w[:npub + 1]), w[npub + 1:], None, draw_blinders=True)
    proofs = [plonk_proof_from_device(cv, pts, evs) for pts, evs in res]
    assert proofs[0] == proofs[1] == proofs[2]
    assert OP.verify(BN254, plonk_vk_from_zkey(z, g["vk_power"]), proofs[0], [ih(x) for x in g["public"]], pairing_product_is_one)
    pk.free()


def check_plonk_rep3_synthetic(ctx, log_n=5, n_public=2, seed=29):
    """Rep3 co-Plonk on the synthetic circuit (additions, empty rows) with random blinder shares: the opened proof
    equals the oracle's plain proof for the summed blinders and is accepted by the verifier."""
    from helpers import plonk_proof_from_device
    from oracle import plonk as OP
    from oracle.pairing_bn254 import pairing_product_is_one
    from workloads.synth_plonk import SynthPlonk
    cv = Conv("bn254")
    syn = SynthPlonk(ctx, log_n, n_public=n_public)
    pk = syn.make_key()
    rng = random.Random(seed)
    bl = [rng.randrange(cv.r) for _ in range(11)]
    res = _plonk_rep3_in_process(ctx, cv, pk, syn.n, syn.key["vk_points"], syn.public_inputs,
                                 syn.full_witness[n_public + 1:], bl)
    proofs = [plonk_proof_from_device(cv, pts, evs) for pts, evs in res]
    assert proofs[0] == proofs[1] == proofs[2]
    assert proofs[0] == OP.prove(syn.oracle_zkey(), syn.full_witness, bl)
    assert OP.verify(BN254, syn.vk_ints(), proofs[0], syn.full_witness[1:n_public + 1], pairing_product_is_one)
    pk.free()


def check_shamir_degree_reduce(ctx, n=64, seed=12):
    """Shamir king-based degree reduction (shamir/network.rs:150-243) assembled from cs_vec_lincomb, for
    n = 3 parties, t = 1: every party masks its degree-2t product share with r_2t, the king interpolates
    with the Lagrange weights, re-shares, and r_t is subtracted -- the result must be a degree-t sharing
    of the products."""
    cv = Conv("bn254")
    r = cv.r
    rng = random.Random(seed)
    nparties, t = 3, 1

    def share(v, deg):
        co = [v] + [rng.randrange(r) for _ in range(deg)]
        return [sum(c * pow(i + 1, e, r) for e, c in enumerate(co)) % r for i in range(nparties)]

    a = [rng.randrange(r) for _ in range(n)]
    b = [rng.randrange(r) for _ in range(n)]
    sa, sb = [share(x, t) for x in a], [share(x, t) for x in b]
    pairs = []
    for _ in range(n):
        rr = rng.randrange(r)
        pairs.append((share(rr, t), share(rr, 2 * t)))
    # lagrange weights for interpolation at 0 from points 1..3
    lam = []
    for i in range(nparties):
        num, den = 1, 1
        for j in range(nparties):
            if j != i:
                num = num * (-(j + 1)) % r
                den = den * ((i + 1) - (j + 1)) % r
        lam.append(num * pow(den, r - 2, r) % r)
    one, minus_one = 1, r - 1
    masked = []
    for p in range(nparties):
        da = ctx.to_device(cv.fr([sa[i][p] for i in range(n)]))
        db = ctx.to_device(cv.fr([sb[i][p] for i in range(n)]))
        dprod = ctx.alloc(n * 32)
        ctx._check(ctx.lib.cs_vec_mul(ctx.h, cv.id, da, db, dprod, n))   # shamir local_mul_vec (arithmetic.rs:73-80)
        d2t = ctx.to_device(cv.fr([pairs[i][1][p] for i in range(n)]))
        dm = ctx.alloc(n * 32)
        ctx.vec_lincomb(cv.id, [dprod, d2t], cv.fr([one, one]), n, dm)   # inp += r_2t
        masked.append(dm)
        for d in (da, db, dprod, d2t):
            ctx.free(d)
    dacc = ctx.alloc(n * 32)
    ctx.vec_lincomb(cv.id, masked, cv.fr(lam), n, dacc)                  # king: sum_j lambda_j * inp_j
    acc = cv.fr_back(ctx.d2h(dacc, (n, 4)))
    # the king sees a*b + r (the double-sharing pair's secret masks the product)
    assert acc == [(x * y + sum(l * pairs[i][1][p] for p, l in enumerate(lam))) % r for i, (x, y) in enumerate(zip(a, b))]
    # fresh degree-t shares of the public value acc: here the trivial re-sharing acc + 0 * x, then share -= r_t
    final = []
    for p in range(nparties):
        drt = ctx.to_device(cv.fr([pairs[i][0][p] for i in range(n)]))
        dout = ctx.alloc(n * 32)
        ctx.vec_lincomb(cv.id, [dacc, drt], cv.fr([one, minus_one]), n, dout)  # share -= r_t
        final.append(cv.fr_back(ctx.d2h(dout, (n, 4))))
        ctx.free(drt)
        ctx.free(dout)
    # opening the degree-t result from parties 1, 2 (weights 2, -1) gives a * b
    for i in range(n):
        assert (2 * final[0][i] - final[1][i]) % r == a[i] * b[i] % r
    for d in masked + [dacc]:
        ctx.free(d)


def check_zkey_ingest(ctx, tmp_path, name="multiplier2"):
    """cs_groth16_pk_from_zkey + cs_wtns_read (co-circom.rs:1005-1016): a snarkjs-format key/witness pair goes
    file -> device and proves to the golden proof bytes; the writer's output is also parsed by the oracle's
    reader, and the reference's own files are ingested too."""
    import os
    import zkey_writer
    from helpers import golden_fixture
    from oracle import formats as OF
    from oracle.formats import proof_to_json
    cv = Conv("bn254")
    z, m, w, g = golden_groth16(name)
    zp, wp = os.path.join(str(tmp_path), name + ".zkey"), os.path.join(str(tmp_path), name + ".wtns")
    zkey_writer.write_zkey(zp, z, m)
    zkey_writer.write_wtns(wp, cv.r, w)
    z2 = OF.read_groth16_zkey(zp)  # the test writer agrees with the oracle's reader
    assert z2["a_query"] == z["a_query"] and OF.zkey_matrices(z2)["a"] == m["a"]
    ref = "Groth16/bn254/%s/" % name
    files = [(zp, wp), (golden_fixture(tmp_path, ref + "circuit.zkey"), golden_fixture(tmp_path, ref + "witness.wtns"))]
    for zf, wf in files:
        pk = B.Groth16Key.from_zkey(ctx, zf)
        assert pk.domain_size() == g["domain_size"] and pk.ni == m["num_instance_variables"]
        wit = B.read_wtns(ctx.lib, wf)
        assert cv.fr_back(wit) == w
        for pr in g["oracle_proofs"]:
            A, Bp, Cp = pk.prove_plain(np.ascontiguousarray(wit[:pk.ni]), np.ascontiguousarray(wit[pk.ni:]),
                                       cv.fr([ih(pr["r"])]), cv.fr([ih(pr["s"])]))
            assert proof_to_json(cv.pt1(A), cv.pt2(Bp), cv.pt1(Cp)) == pr["json"]
        pk.free()
    # error behaviour
    bad = os.path.join(str(tmp_path), "bad.zkey")
    open(bad, "wb").write(b"nope" + bytes(20))
    try:
        B.Groth16Key.from_zkey(ctx, bad)
        raise AssertionError("bad magic must fail")
    except B.CsError as e:
        assert "bad magic" in str(e)


def check_prove_cli(ctx_lib_path, tmp_path, name="multiplier2"):
    """python -m co_snarks_b200.prove: zkey + wtns in, snarkjs-layout proof.json out, accepted by the pairing
    check under the fixture's verification key (the acceptance test of co-groth16/src/lib.rs:40-91)."""
    import json
    import os
    import zkey_writer
    from co_snarks_b200 import prove as P
    from oracle.formats import read_proof_json
    cv = Conv("bn254")
    z, m, w, g = golden_groth16(name)
    zp, wp = os.path.join(str(tmp_path), "c.zkey"), os.path.join(str(tmp_path), "w.wtns")
    zkey_writer.write_zkey(zp, z, m)
    zkey_writer.write_wtns(wp, cv.r, w)
    out, pub = os.path.join(str(tmp_path), "proof.json"), os.path.join(str(tmp_path), "public.json")
    argv = ["--zkey", zp, "--wtns", wp, "--out", out, "--public-out", pub]
    if ctx_lib_path:
        argv += ["--lib", ctx_lib_path]
    P.main(argv)
    proof = read_proof_json(out)
    public = [int(x) for x in json.load(open(pub))]
    assert public == [ih(x) for x in g["public"]]
    assert groth16_verify(OG.vk_from_zkey(z), public, proof)
    assert json.load(open(out))["protocol"] == "groth16"


def check_prove_cli_rep3_shares(ctx_lib_path, tmp_path, name="multiplier2"):
    """The CLI in Rep3 mode: three share files (the bincode layout co-circom split-witness writes; party 1's previous
    half given as a seed to exercise the compressed variant) in, one opened proof out, accepted under the fixture's
    verification key -- tests/tests/circom/e2e_tests/rep3.rs:36-137 from files."""
    import json
    import os
    import zkey_writer
    from co_snarks_b200 import prove as P
    from oracle.formats import read_proof_json
    cv = Conv("bn254")
    r = cv.r
    z, m, w, g = golden_groth16(name)
    ni = m["num_instance_variables"]
    zp = os.path.join(str(tmp_path), "c3.zkey")
    zkey_writer.write_zkey(zp, z, m)
    wsh = OG.share_rep3(w[ni:], r, random.Random(61))
    paths = []
    for i in range(3):
        pth = os.path.join(str(tmp_path), "shares.%d" % i)
        write_rep3_share_file(pth, w[:ni], 0, wsh[i], r)
        paths.append(pth)
    out, pub = os.path.join(str(tmp_path), "proof3.json"), os.path.join(str(tmp_path), "public3.json")
    argv = ["--zkey", zp, "--rep3-shares"] + paths + ["--out", out, "--public-out", pub]
    if ctx_lib_path:
        argv += ["--lib", ctx_lib_path]
    P.main(argv)
    public = [int(x) for x in json.load(open(pub))]
    assert public == [ih(x) for x in g["public"]]
    assert groth16_verify(OG.vk_from_zkey(z), public, read_proof_json(out))
    # the compressed form: additive shares (variant 2), replicated by one reshare inside the CLI
    paths2 = []
    for i in range(3):
        pth = os.path.join(str(tmp_path), "add_shares.%d" % i)
        write_rep3_share_file(pth, w[:ni], 2, [ab[0] for ab in wsh[i]], r)
        paths2.append(pth)
    out2 = os.path.join(str(tmp_path), "proof3b.json")
    argv = ["--zkey", zp, "--rep3-shares"] + paths2 + ["--out", out2]
    if ctx_lib_path:
        argv += ["--lib", ctx_lib_path]
    P.main(argv)
    assert groth16_verify(OG.vk_from_zkey(z), public, read_proof_json(out2))


def check_prove_cli_plonk(ctx_lib_path, tmp_path, name="multiplier2"):
    """The same CLI on a Plonk zkey: snarkjs-layout Plonk proof.json accepted by Plonk::verify (plonk.rs:110-245)."""
    import json
    import os
    import zkey_writer
    from co_snarks_b200 import prove as P
    from helpers import golden_plonk, plonk_vk_from_zkey
    from oracle import plonk as OP
    from oracle.formats import read_plonk_proof_json
    from oracle.pairing_bn254 import pairing_product_is_one
    cv = Conv("bn254")
    z, w, g = golden_plonk(name)
    zp, wp = os.path.join(str(tmp_path), "p.zkey"), os.path.join(str(tmp_path), "pw.wtns")
    zkey_writer.write_plonk_zkey(zp, z)
    zkey_writer.write_wtns(wp, cv.r, w)
    out, pub = os.path.join(str(tmp_path), "plonk_proof.json"), os.path.join(str(tmp_path), "plonk_public.json")
    argv = ["--zkey", zp, "--wtns", wp, "--out", out, "--public-out", pub]
    if ctx_lib_path:
        argv += ["--lib", ctx_lib_path]
    P.main(argv)
    public = [int(x) for x in json.load(open(pub))]
    assert public == [ih(x) for x in g["public"]]
    assert OP.verify(BN254, plonk_vk_from_zkey(z, g["vk_power"]), read_plonk_proof_json(out), public, pairing_product_is_one)
    assert json.load(open(out))["protocol"] == "plonk"


def check_libsnark_reduction(ctx, m_vars=50, seed=14):
    """LibSnarkReduction::witness_map_from_matrices (reduction.rs:241-342), plain and Rep3, against the oracle
    restatement; the oracle itself is checked by the QAP identity A(x)B(x) - C(x) = H(x) Z(x) at a random point
    (the reference's only fixtures for this reduction are BLS12-377 keys, a curve outside the GPU build)."""
    from oracle.ntt import ifft
    cv = Conv("bn254")
    r = cv.r
    rng = random.Random(seed)
    w = [1, rng.randrange(r)]
    A, Bm, Cm = [], [], []
    for k in range(2, m_vars):
        j1, j2, j3 = rng.randrange(k), rng.randrange(k), rng.randrange(k)
        A.append([(1, j1), (1, j2)] if j1 != j2 else [(2, j1)])
        Bm.append([(rng.randrange(1, 9), j3)])
        Cm.append([(Bm[-1][0][0], k)])
        w.append((w[j1] + w[j2]) * w[j3] % r)
    mat = dict(a=A, b=Bm, c=Cm, num_constraints=m_vars - 2, num_instance_variables=2, num_witness_variables=m_vars - 2)
    h = OG.witness_map_libsnark(mat, w[:2], w[2:], r)
    n, gen, g = OG.ark_domain(m_vars, r)
    a = OG.evaluate_constraint_plain(A, w[:2], w[2:], n, r)
    a[m_vars - 2:m_vars] = w[:2]
    b = OG.evaluate_constraint_plain(Bm, w[:2], w[2:], n, r)
    c = OG.evaluate_constraint_plain(Cm, w[:2], w[2:], n, r)
    x = rng.randrange(r)
    ev = lambda p: sum(co * pow(x, i, r) for i, co in enumerate(p)) % r
    assert (ev(ifft(a, gen, r)) * ev(ifft(b, gen, r)) - ev(ifft(c, gen, r))) % r == ev(h) * (pow(x, n, r) - 1) % r
    # device: key with dummy points (only the matrices matter for the witness map)
    G = og1(BN254)
    P1 = cv.g1([BN254.g1])
    P2 = cv.g2([BN254.g2])
    mc = dict(num_constraints=m_vars - 2, num_instance_variables=2, num_witness_variables=m_vars - 2,
              a=cv.csr(A), b=cv.csr(Bm), c=cv.csr(Cm))
    pts = dict(alpha_g1=P1, beta_g1=P1, beta_g2=P2, delta_g1=P1, delta_g2=P2, a_query=np.repeat(P1, m_vars, 0),
               b_g1_query=np.repeat(P1, m_vars, 0), b_g2_query=np.repeat(P2, m_vars, 0),
               l_query=np.repeat(P1, m_vars - 2, 0), h_query=np.repeat(P1, n, 0))
    pk = B.Groth16Key(ctx, cv.id, mc, pts)
    assert pk.domain_size() == n
    pub = cv.fr(w[:2])
    assert cv.fr_back(pk.witness_map_libsnark(pub, cv.fr(w[2:]))) == h
    wsh = OG.share_rep3(w[2:], r, rng)
    prf = [[rng.randrange(r) for _ in range(n)] for _ in range(3)]
    masks = [[(prf[i][j] - prf[(i + 2) % 3][j]) % r for j in range(n)] for i in range(3)]
    tot = [0] * n
    for i in range(3):
        sh = cv.fr([v for ab in wsh[i] for v in ab])
        got = cv.fr_back(pk.witness_map_libsnark(pub, sh, B.CS_REP3, i, cv.fr(masks[i])))
        assert got == OG.witness_map_libsnark(mat, w[:2], wsh[i], r, "rep3", i, masks[i])
        tot = [(p + q) % r for p, q in zip(tot, got)]
    assert tot == h
    pk.free()


def check_rep3_batch_ops(ctx, n=257, seed=31):
    """The batched VM opcodes (circom-mpc-vm/src/mpc/batched_rep3.rs:124-188, 322-337) on all three parties'
    share vectors: every op's result, opened, equals the plain operation on the secrets; the per-party placement of
    public operands follows arithmetic.rs:41-48 and promote_to_trivial_share (arithmetic.rs:321-327) exactly."""
    from oracle import groth16 as OG
    cv = Conv("bn254")
    r = cv.r
    rng = random.Random(seed)
    xs = [rng.randrange(r) for _ in range(n)]
    ys = [rng.randrange(r) for _ in range(n)]
    pub = [rng.randrange(r) for _ in range(n)]
    xsh, ysh = OG.share_rep3(xs, r, rng), OG.share_rep3(ys, r, rng)
    flat = lambda sh: cv.fr([v for ab in sh for v in ab])
    dx = [ctx.to_device(flat(xsh[i])) for i in range(3)]
    dy = [ctx.to_device(flat(ysh[i])) for i in range(3)]
    dp = ctx.to_device(cv.fr(pub))
    do = [ctx.alloc(n * 64) for _ in range(3)]
    cases = [(B.R3B_ADD, True, lambda x, y, p: (x + y) % r), (B.R3B_SUB, True, lambda x, y, p: (x - y) % r),
             (B.R3B_ADD_PUBLIC, False, lambda x, y, p: (x + p) % r), (B.R3B_SUB_PUBLIC, False, lambda x, y, p: (x - p) % r),
             (B.R3B_PUBLIC_SUB, False, lambda x, y, p: (p - x) % r), (B.R3B_MUL_PUBLIC, False, lambda x, y, p: x * p % r),
             (B.R3B_NEG, None, lambda x, y, p: (-x) % r), (B.R3B_PROMOTE, "promote", lambda x, y, p: p)]
    for op, second, expect in cases:
        outs = []
        for i in range(3):
            d_y = dy[i] if second is True else (None if second is None else dp)
            d_x = None if second == "promote" else dx[i]
            ctx.rep3_batch(cv.id, op, i, d_x, d_y, do[i], n)
            outs.append(cv.fr_back(ctx.d2h(do[i], (2 * n, 4))))
        for k in range(n):
            # replicated: party i's b is party i-1's a; the three a's open to the expected value
            assert all(outs[i][2 * k + 1] == outs[(i + 2) % 3][2 * k] for i in range(3)), (op, k)
            assert sum(outs[i][2 * k] for i in range(3)) % r == expect(xs[k], ys[k], pub[k]), (op, k)
        if op == B.R3B_ADD_PUBLIC:  # the public value sits in party 0's a (= party 1's b) and nowhere else
            assert outs[2][0] == xsh[2][0][0] and outs[2][1] == xsh[2][0][1]
            assert outs[0][0] == (xsh[0][0][0] + pub[0]) % r and outs[0][1] == xsh[0][0][1]
        if op == B.R3B_PROMOTE:
            assert (outs[0][0], outs[0][1]) == (pub[0], 0) and (outs[1][0], outs[1][1]) == (0, pub[0]) and outs[2][:2] == [0, 0]
    # open (open_vec): b-components travel to the next party, a + b + c
    recv = [ctx.alloc(n * 32) for _ in range(3)]
    lib = ctx.lib
    for i in range(3):
        ctx._check(lib.cs_rep3_batch_open_send(ctx.h, cv.id, dx[i], n, recv[(i + 1) % 3]))
    ctx.synchronize()
    for i in range(3):
        ctx._check(lib.cs_rep3_batch_open_finish(ctx.h, cv.id, dx[i], recv[i], do[i], n))
        assert cv.fr_back(ctx.d2h(do[i], (n, 4))) == xs
    for d in dx + dy + do + recv + [dp]:
        ctx.free(d)


def check_honk_commit_batch(ctx, n=200, seed=41):
    """CoUtils::commit over the Ignition CRS (co-noir-common/src/lib.rs:88-101 -> fast_msm, honk_curve.rs:81-83) for a
    round of polynomials at once: plain commitments == oracle MSM; Rep3 commitments are the point share {a, b} of
    co-noir-common/src/mpc/rep3.rs:259-266 and the three parties' a-points open to the plain commitment; shorter
    polynomials use the leading CRS points only."""
    from oracle import groth16 as OG
    cv = Conv("bn254")
    r = cv.r
    g = load_golden("crs_bn254_g1_first1024")
    pts = [gp1(P) for P in g["points"]][:n]
    crs = ctx.bases_upload(cv.id, 0, cv.g1(pts))
    rng = random.Random(seed)
    G = og1(BN254)
    lens = [n, n - 17, 5, 0]
    polys = [[rng.randrange(r) for _ in range(l)] for l in lens]
    d = [ctx.to_device(cv.fr(p)) if p else 0 for p in polys]
    out = ctx.honk_commit_batch(crs, B.CS_PLAIN, d, lens)
    exp = [G.msm(pts[:l], p) if l else None for p, l in zip(polys, lens)]
    assert [cv.pt1(o) for o in out] == exp
    # Rep3: two polynomials, every party commits to both components
    sh = [OG.share_rep3(p, r, rng) for p in polys[:2]]
    a_pts = [[None] * 2 for _ in range(3)]
    for i in range(3):
        ds = [ctx.to_device(cv.fr([v for ab in sh[k][i] for v in ab])) for k in range(2)]
        o = ctx.honk_commit_batch(crs, B.CS_REP3, ds, lens[:2])
        for k in range(2):
            a_pts[i][k], b_pt = cv.pt1(o[2 * k]), cv.pt1(o[2 * k + 1])
            assert a_pts[i][k] == G.msm(pts[:lens[k]], [ab[0] for ab in sh[k][i]])
            assert b_pt == G.msm(pts[:lens[k]], [ab[1] for ab in sh[k][i]])
        for x in ds:
            ctx.free(x)
    for k in range(2):
        acc = None
        for i in range(3):
            acc = G.add(acc, a_pts[i][k])
        assert acc == exp[k]
    with pytest.raises(RuntimeError):
        ctx.honk_commit_batch(crs, B.CS_PLAIN, [d[0]], [n + 1])  # longer than the CRS
    for x in d:
        if x:
            ctx.free(x)
    crs.free()


def check_share_rep3_device(ctx, n=1000):
    """rep3::share_field_elements on the device (rep3.rs:281-293): the three parties' vectors are replicated shares
    of the witness (a + b + c = value; party i's b is party i-1's a), uniform draws stay below r, a fixed seed is
    reproducible and two seeds differ; cs_fr_rand_device: exact rejection sampling on per-element sub-streams."""
    cv = Conv("bn254")
    r = cv.r
    rng = random.Random(9)
    vals = [rng.randrange(r) for _ in range(n)]
    lib = ctx.lib
    dw = ctx.to_device(cv.fr(vals))
    ds = [ctx.alloc(n * 64) for _ in range(3)]
    seed = bytes(range(32))
    ctx._check(lib.cs_share_rep3_device(ctx.h, cv.id, dw, n, seed, ds[0], ds[1], ds[2]))
    sh = [cv.fr_back(ctx.d2h(d, (2 * n, 4))) for d in ds]
    for k in range(n):
        assert sum(sh[i][2 * k] for i in range(3)) % r == vals[k]
        assert all(sh[i][2 * k + 1] == sh[(i + 2) % 3][2 * k] for i in range(3))
    first = sh[0][:8]
    ctx._check(lib.cs_share_rep3_device(ctx.h, cv.id, dw, n, seed, ds[0], ds[1], ds[2]))
    assert cv.fr_back(ctx.d2h(ds[0], (2 * n, 4)))[:8] == first
    ctx._check(lib.cs_share_rep3_device(ctx.h, cv.id, dw, n, None, ds[0], ds[1], ds[2]))  # OS entropy
    assert cv.fr_back(ctx.d2h(ds[0], (2 * n, 4)))[:8] != first
    # the raw limbs of a uniform draw are a 254-bit value below r; the first draw of sub-stream 0 matches the host's
    # ChaCha12 block function (cs_chacha_keystream with stream id 0 = the plain keystream)
    dr = ctx.alloc(n * 32)
    ctx._check(lib.cs_fr_rand_device(ctx.h, cv.id, seed, 0, dr, n))
    raw = ctx.d2h(dr, (n, 4))
    ints = B.limbs_to_ints(raw)
    assert all(v < r for v in ints) and len(set(ints)) == n
    ks = np.asarray(ctx.chacha_keystream(seed, 0, 12, 4), dtype=np.uint32).reshape(-1)
    for half in range(8):
        w = ks[8 * half:8 * half + 8]
        limbs = [int(w[2 * i]) | (int(w[2 * i + 1]) << 32) for i in range(4)]
        limbs[3] &= (1 << 62) - 1
        v = sum(l << (64 * i) for i, l in enumerate(limbs))
        if v < r:
            assert ints[0] == v
            break
    for d in ds + [dw, dr]:
        ctx.free(d)


def write_rep3_share_file(path, public_ints, variant, payload, r):
    """TEST-SIDE writer of the CompressedRep3SharedWitness bincode layout (see include/cosnarks_gpu.h):
    variant 0: payload = [(a, b), ...]; 2: [x, ...]; 1: (seeded_a, seeded_b); 3: seeded, where seeded is either
    ("shares", [x, ...]) or ("seed", seed32, length)."""
    import struct

    def ark_vec(elems, width):
        body = struct.pack("<Q", len(elems)) + b"".join(int(e).to_bytes(32, "little") if width == 1 else
                                                        b"".join(int(x).to_bytes(32, "little") for x in e) for e in elems)
        return struct.pack("<Q", len(body)) + body

    def seeded(sd):
        if sd[0] == "shares":
            return struct.pack("<I", 0) + ark_vec(sd[1], 1)
        return struct.pack("<I", 1) + bytes(sd[1]) + struct.pack("<Q", sd[2])
    out = ark_vec(public_ints, 1) + struct.pack("<I", variant)
    if variant == 0:
        out += ark_vec(payload, 2)
    elif variant == 2:
        out += ark_vec(payload, 1)
    elif variant == 1:
        out += seeded(payload[0]) + seeded(payload[1])
    else:
        out += seeded(payload)
    with open(path, "wb") as f:
        f.write(out)


def check_rep3_share_files(lib, tmp_path):
    """cs_rep3_witness_read on all four Rep3ShareVecType variants (co-circom-types/src/lib.rs:162-219): replicated,
    seeded replicated (one half given as a seed: expanded with F::rand over ChaCha12), additive, seeded additive;
    malformed files give an error code."""
    import os
    cv = Conv("bn254")
    r = cv.r
    rng = random.Random(3)
    pub = [1, rng.randrange(r)]
    n = 50
    rep = [(rng.randrange(r), rng.randrange(r)) for _ in range(n)]
    p = os.path.join(str(tmp_path), "w.shared")
    write_rep3_share_file(p, pub, 0, rep, r)
    gp, gs, kind = B.read_rep3_witness(lib, p, cv.id)
    assert kind == B.CS_REP3 and cv.fr_back(gp) == pub and cv.fr_back(gs) == [x for ab in rep for x in ab]
    add = [rng.randrange(r) for _ in range(n)]
    write_rep3_share_file(p, pub, 2, add, r)
    gp, gs, kind = B.read_rep3_witness(lib, p, cv.id)
    assert kind == B.CS_PLAIN and cv.fr_back(gs) == add
    seed = bytes(range(7, 39))
    write_rep3_share_file(p, pub, 3, ("seed", seed, n), r)
    _, seeded_vals, kind = B.read_rep3_witness(lib, p, cv.id)
    seeded_ints = B.limbs_to_ints(seeded_vals)  # F::rand output limbs are the Montgomery representation
    assert kind == B.CS_PLAIN and len(seeded_ints) == n and all(v < r for v in seeded_ints) and len(set(seeded_ints)) == n
    write_rep3_share_file(p, pub, 1, (("seed", seed, n), ("shares", add)), r)
    _, gs, kind = B.read_rep3_witness(lib, p, cv.id)
    assert kind == B.CS_REP3
    assert (gs[:, :4] == seeded_vals).all() and cv.fr_back(gs[:, 4:]) == add
    # error behaviour: length mismatch between the two halves, a non-canonical element, truncation
    write_rep3_share_file(p, pub, 1, (("seed", seed, n - 1), ("shares", add)), r)
    with pytest.raises(RuntimeError, match="Lengths of shares do not match"):
        B.read_rep3_witness(lib, p, cv.id)
    write_rep3_share_file(p, pub, 2, [r] + add[1:], r)
    with pytest.raises(RuntimeError):
        B.read_rep3_witness(lib, p, cv.id)
    data = open(p, "rb").read()
    open(p, "wb").write(data[:-5])
    with pytest.raises(RuntimeError):
        B.read_rep3_witness(lib, p, cv.id)


def check_sumcheck(ctx, log_n=5, seed=51, curve="bn254"):
    """UltraHonk sumcheck kernels (csrc/cs_sumcheck.cuh) against oracle/sumcheck.py, plain and 3-party Rep3, and through
    a whole sumcheck of the arithmetic relation: S_0(0) + S_0(1) = sum over the hypercube, S_i(0) + S_i(1) =
    S_{i-1}(u_{i-1}), and the last claim equals the relation on the fully folded polynomials."""
    from oracle import chacha as OC
    from oracle import groth16 as OG
    from oracle import sumcheck as OS
    cv = Conv(curve)
    r = cv.r
    rng = random.Random(seed)
    n = 1 << log_n
    names_w, names_q = OS.ARITH_WITNESS, OS.ARITH_SELECTORS
    # ---- gate separator
    betas = [rng.randrange(r) for _ in range(log_n)]
    d_beta = ctx.alloc(n * 32)
    ctx.sumcheck_gate_separator(cv.id, cv.fr(betas), d_beta)
    beta_products = OS.gate_separator(betas, log_n, r)
    assert cv.fr_back(ctx.d2h(d_beta, (n, 4))) == beta_products
    d_one = ctx.alloc(32)
    ctx.sumcheck_gate_separator(cv.id, cv.fr([]), d_one)  # log_n = 0: the single entry 1
    assert cv.fr_back(ctx.d2h(d_one, (1, 4))) == [1]
    ctx.free(d_one)
    # ---- polynomials: q_arith takes every branch value (0 disables an edge entirely when both rows are 0)
    polys = {nm: [rng.randrange(r) for _ in range(n)] for nm in names_w + names_q}
    polys["q_arith"] = [rng.choice([0, 0, 1, 2, 3, 4, rng.randrange(r)]) for _ in range(n)]
    polys["q_arith"][0:2] = [0, 0]
    polys["q_arith"][6:8] = [0, 0]
    shares = {nm: OG.share_rep3(polys[nm], r, rng) for nm in names_w}  # [party][row] -> (a, b)
    flat = lambda sh: cv.fr([v for ab in sh for v in ab])
    bufs = []

    def dev(arr):
        p = ctx.to_device(arr)
        bufs.append(p)
        return p
    d_plain = {nm: dev(cv.fr(polys[nm])) for nm in names_w + names_q}
    d_party = [dict({nm: dev(flat(shares[nm][i])) for nm in names_w}, **{nm: d_plain[nm] for nm in names_q}) for i in range(3)]

    # ---- one round, plain and Rep3, against the oracle (periodicity 2 = first round)
    r0, r1 = ctx.sumcheck_arith_round(cv.id, B.CS_PLAIN, 0, d_plain, n, d_beta, 2)
    exp0, exp1 = OS.arith_round_plain(polys, n, beta_products, 2, r)
    assert cv.fr_back(r0) == exp0 and cv.fr_back(r1) == exp1
    seeds = [bytes((11 * p + i) & 0xff for i in range(32)) for p in range(3)]
    pos = [5, 64, 19]
    tot0, tot0m, tot1 = [0] * 6, [0] * 6, [0] * 5
    views = []
    for i in range(3):
        view = dict({nm: shares[nm][i] for nm in names_w}, **{nm: polys[nm] for nm in names_q})
        e0, e1 = OS.arith_round_rep3(view, i, n, beta_products, 2, r)
        g0, g1 = ctx.sumcheck_arith_round(cv.id, B.CS_REP3, i, d_party[i], n, d_beta, 2)
        g1 = cv.fr_back(g1)
        assert cv.fr_back(g0) == e0, i
        assert [(g1[2 * k], g1[2 * k + 1]) for k in range(5)] == e1, i
        views.append(e1)
        tot0 = [(a + b) % r for a, b in zip(tot0, e0)]
        tot1 = [(a + b[0]) % r for a, b in zip(tot1, e1)]
        # with the zero-share masks drawn from the party's two streams
        prev = (i + 2) % 3
        prf = B.Rep3Prf((C.c_uint8 * 32)(*seeds[i]), pos[i], (C.c_uint8 * 32)(*seeds[prev]), pos[prev], 12)
        m0, _ = ctx.sumcheck_arith_round(cv.id, B.CS_REP3, i, d_party[i], n, d_beta, 2, prf)
        m0 = cv.fr_back(m0)
        masks = OC.masking_field_elements_vec(seeds[i], pos[i], seeds[prev], pos[prev], 6, r)
        assert m0 == [(a + b) % r for a, b in zip(e0, masks)], i
        tot0m = [(a + b) % r for a, b in zip(tot0m, m0)]
    assert tot0 == exp0 and tot0m == exp0 and tot1 == exp1  # the parties' accumulators open to the plain ones
    assert all(views[i][k][1] == views[(i + 2) % 3][k][0] for i in range(3) for k in range(5))  # r1 stays replicated

    # ---- Shamir(3, 1) parties run the PLAIN kernel on their degree-t shares (co-noir-common/src/mpc/shamir.rs: public
    # values are added by every party, products are local and raise the degree): r0 comes out as a degree-2t sharing
    # (what degree_reduce takes next), r1 as a degree-t sharing
    def shamir_share(vals, t=1, nparties=3):
        out = [[] for _ in range(nparties)]
        for v in vals:
            co = [v] + [rng.randrange(r) for _ in range(t)]
            for i in range(nparties):
                out[i].append(sum(c * pow(i + 1, k, r) for k, c in enumerate(co)) % r)
        return out
    sh_sh = {nm: shamir_share(polys[nm]) for nm in names_w}
    got = []
    for i in range(3):
        d_sh = dict({nm: dev(cv.fr(sh_sh[nm][i])) for nm in names_w}, **{nm: d_plain[nm] for nm in names_q})
        g0, g1 = ctx.sumcheck_arith_round(cv.id, B.CS_PLAIN, 0, d_sh, n, d_beta, 2)
        got.append((cv.fr_back(g0), cv.fr_back(g1)))
    lag3 = [_lagrange_basis_at(xs_=[1, 2, 3], i=i, x=0, r=r) for i in range(3)]   # 2t + 1 = 3 points: degree 2t
    lag2 = [_lagrange_basis_at(xs_=[1, 2], i=i, x=0, r=r) for i in range(2)]      # t + 1 = 2 points: degree t
    assert [sum(l * got[i][0][k] for i, l in enumerate(lag3)) % r for k in range(6)] == exp0
    assert [sum(l * got[i][1][k] for i, l in enumerate(lag2)) % r for k in range(5)] == exp1
    assert [sum(l * got[i + 1][1][k] for i, l in enumerate(
        [_lagrange_basis_at(xs_=[2, 3], i=j, x=0, r=r) for j in range(2)])) % r for k in range(5)] == exp1

    # ---- fold: public + shared batches against the oracle, down to one row (+ the zero the reference pushes)
    u0 = rng.randrange(r)
    for shared in (False, True):
        nms = names_w if shared else names_q
        cur = {nm: (shares[nm][1] if shared else polys[nm]) for nm in nms}
        d_cur = {nm: (d_party[1][nm] if shared else d_plain[nm]) for nm in nms}
        length, u = n, u0
        comps = 2 if shared else 1
        while length >= 2:
            d_out = {nm: ctx.alloc(max(length // 2, 2) * 32 * comps) for nm in nms}
            ctx.sumcheck_fold(cv.id, [d_cur[nm] for nm in nms], [d_out[nm] for nm in nms], shared, length, cv.fr([u])[0])
            for nm in nms:
                cur[nm] = OS.partially_evaluate(cur[nm][:length], u, r)
                got = cv.fr_back(ctx.d2h(d_out[nm], (len(cur[nm]) * comps, 4)))
                want = [v for ab in cur[nm] for v in ab] if shared else cur[nm]
                assert got == want, (nm, length)
            bufs.extend(d_out.values())
            d_cur, length, u = d_out, length // 2, (u * 7 + 3) % r

    # ---- the whole sumcheck of this relation on the plain polynomials
    alpha = rng.randrange(r)
    neg_half = (-pow(2, -1, r)) % r

    def relation_row(x):  # q_arith * [...] + alpha * q_arith (q_arith - 1)(q_arith - 2)(...)   (the doc comment, :270-320)
        qa = x["q_arith"]
        f0 = (x["w_l"] * x["w_r"] % r * x["q_m"] % r * (qa - 3) % r * neg_half + x["q_l"] * x["w_l"] + x["q_r"] * x["w_r"]
              + x["q_o"] * x["w_o"] + x["q_4"] * x["w_4"] + x["q_c"] + (qa - 1) * x["w_4_shift"]) % r * qa % r
        f1 = (x["w_l"] + x["w_4"] - x["w_l_shift"] + x["q_m"]) % r * (qa - 2) % r * (qa - 1) % r * qa % r
        return (f0 + alpha * f1) % r

    def eval_univariate(evals, x):
        return sum(v * _lagrange_basis(len(evals), i, x, r) for i, v in enumerate(evals)) % r
    target = sum(relation_row({nm: polys[nm][j] for nm in polys}) * beta_products[j] for j in range(n)) % r
    cur = dict(polys)
    d_cur = dict(d_plain)
    size, periodicity, partial, us = n, 2, 1, []
    SIZE = 8  # BATCHED_RELATION_PARTIAL_LENGTH
    for rnd in range(log_n):
        g0, g1 = ctx.sumcheck_arith_round(cv.id, B.CS_PLAIN, 0, d_cur, size, d_beta, periodicity)
        g0, g1 = cv.fr_back(g0), cv.fr_back(g1)
        assert (g0, g1) == OS.arith_round_plain({nm: cur[nm][:size] for nm in cur}, size, beta_products, periodicity, r)
        S = OS.batch_univariates(g0, g1, alpha, betas[rnd], partial, SIZE, r)
        assert (S[0] + S[1]) % r == target, rnd
        u = rng.randrange(r)
        us.append(u)
        target = eval_univariate(S, u)
        partial = partial * (1 + u * (betas[rnd] - 1)) % r  # GateSeparatorPolynomial::partially_evaluate (types.rs:96-102)
        periodicity *= 2
        nms = list(cur)
        d_out = {nm: ctx.alloc(max(size // 2, 2) * 32) for nm in nms}
        ctx.sumcheck_fold(cv.id, [d_cur[nm] for nm in nms], [d_out[nm] for nm in nms], False, size, cv.fr([u])[0])
        bufs.extend(d_out.values())
        d_cur = d_out
        cur = {nm: OS.partially_evaluate(cur[nm][:size], u, r) for nm in nms}
        size //= 2
    final = {nm: cv.fr_back(ctx.d2h(d_cur[nm], (1, 4)))[0] for nm in cur}
    assert final == {nm: cur[nm][0] for nm in cur}
    assert target == relation_row(final) * partial % r  # the claim the verifier checks against the opened evaluations
    for p in bufs + [d_beta]:
        ctx.free(p)


def _lagrange_basis(n, i, x, r):
    num, den = 1, 1
    for j in range(n):
        if j != i:
            num = num * (x - j) % r
            den = den * (i - j) % r
    return num * pow(den, -1, r) % r


def _lagrange_basis_at(xs_, i, x, r):
    num, den = 1, 1
    for j, xj in enumerate(xs_):
        if j != i:
            num = num * (x - xj) % r
            den = den * (xs_[i] - xj) % r
    return num * pow(den, -1, r) % r
