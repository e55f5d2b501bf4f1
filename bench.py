#!/usr/bin/env python
"""bench.py -- Groth16 proofs/s on the co-snarks hot path (BASELINE.json metric), B200.

A "step" = one Groth16 proof over BN254 for a synthetic 2^20-constraint R1CS (BASELINE.json
configs[1]: plain prover, 1xB200): witness map (2 SpMV, 6 NTT of 2^20, 3 element kernels) + 5 MSMs
(4 G1 + 1 G2 of ~2^20) + assembly, through the reference-facing C ABI (cs_groth16_prove_plain).
  value : proofs/s with the witness already resident in HBM (cs_groth16_prove_plain_device), CUDA events
  e2e   : the same through host (pinned) buffers -- H2D of the witness and D2H of the results inside
          the timed region, wall clock between synchronisations
  N > 1 : N independent prover replicas, one per GPU (the path shards by proof; no data-path
          collective), barrier + max over ranks, value = N*K / t      ("scaling": "weak")
  --impl reference : the oracle's C restatement of the reference CPU path (oracle/c) on the host cores.
Prints ONE JSON line on rank 0.

oracle/ is used here only as the checker and the CPU baseline, never inside a timed region and never by the
product: before timing, rank 0 has the oracle's pairing verifier accept one GPU proof (the "proof
pairing-verified" flag in `data`), and the cpu_baseline / --impl reference legs time oracle/c on the host.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ next to the sources

# the prover uses more streams than the driver's default 8 hardware queues (see csrc/cs_api.cu); must be set before the
# CUDA context exists
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "co-Groth16 proofs/sec (BN254, 2^20 constraints); MSM Mscalar/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons = [], None, set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                smax = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def _rep3_shares(ctx, syn, cvid):
    """Replicated sharing of the private witness (rep3.rs:281-293): x = x0 + x1 + x2, party i holds (x_i, x_{i-1}).
    Deterministic (PCG64 seed 5) so that every rank derives the same sharing without communication."""
    import numpy as np
    from co_snarks_b200.rep3 import random_field_limbs
    lib = ctx.lib
    share_rng = np.random.Generator(np.random.PCG64(5))
    nw = syn.private_witness.shape[0]
    x0, x1 = random_field_limbs(share_rng, nw), random_field_limbs(share_rng, nw)
    d0, d1, dw = ctx.to_device(x0), ctx.to_device(x1), ctx.to_device(syn.private_witness)
    ctx._check(lib.cs_vec_sub(ctx.h, cvid, dw, d0, dw, nw))
    ctx._check(lib.cs_vec_sub(ctx.h, cvid, dw, d1, dw, nw))
    x2 = ctx.d2h(dw, (nw, 4))
    for d in (d0, d1, dw):
        ctx.free(d)
    return (x0, x1, x2)


def _party_shares(xs, pid, pinned=True):
    import numpy as np
    import torch
    sh = np.ascontiguousarray(np.concatenate([xs[pid], xs[(pid + 2) % 3]], axis=1))
    if not pinned:
        return sh
    t = torch.empty(sh.shape, dtype=torch.int64).pin_memory()
    t.numpy().view(np.uint64)[:] = sh
    return t.numpy().view(np.uint64), t


def _verify_proof(syn, proof):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import Conv
    from oracle.pairing_bn254 import groth16_verify
    cv = Conv("bn254")
    return bool(groth16_verify(syn.vk_ints(), syn.witness[1:2], (cv.pt1(proof[0]), cv.pt2(proof[1]), cv.pt1(proof[2]))))


def rep3_threads_one_gpu(args, ctx, pk, syn):
    """BASELINE's metric config (co-Groth16, 3-party Rep3, 2^20) when only ONE GPU is available: the three parties
    run as three host threads sharing the GPU, each with its own context, device-resident key and streams, the
    whole protocol inside the library (cs_groth16_rep3_prove) over in-process mailbox nets."""
    import threading
    import numpy as np
    import torch
    from co_snarks_b200 import binding as B
    lib = ctx.lib
    t0 = time.time()
    ctxs = [ctx] + [B.Context(ctx.device) for _ in range(2)]
    pks = [pk] + [B.Groth16Key(c, B.CS_BN254, syn.matrices, syn.points, args.window_bits) for c in ctxs[1:]]
    key_s = time.time() - t0
    xs = _rep3_shares(ctx, syn, B.CS_BN254)
    host_sh = [_party_shares(xs, i) for i in range(3)]
    dev_sh = [ctxs[i].to_device(host_sh[i][0]) for i in range(3)]
    nets0 = [B.Net.peer(ctxs[i], i, 3) for i in range(3)]
    nets1 = [B.Net.peer(ctxs[i], i, 3) for i in range(3)]
    for i in range(3):
        nets0[i].connect_local(nets0)
        nets1[i].connect_local(nets1)
    seeds = [B.os_random(lib, 32) for _ in range(3)]
    states = [B.Rep3StateC.from_seeds(lib, i, seeds[i], seeds[(i + 2) % 3]) for i in range(3)]
    pub = syn.public_inputs

    def run(steps, device):
        res, errs = {}, []
        bar = threading.Barrier(3)

        def party(i):
            try:
                bar.wait()
                for _ in range(steps):
                    res[i] = pks[i].rep3_prove(nets0[i], nets1[i], states[i], pub,
                                               None if device else host_sh[i][0], dev_sh[i] if device else None)
            except Exception as e:  # noqa: BLE001
                errs.append(e)
                bar.abort()
        th = [threading.Thread(target=party, args=(i,)) for i in range(3)]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        torch.cuda.synchronize()
        if errs:
            raise errs[0]
        return (time.perf_counter() - t0) * 1e3, res
    _, res = run(1, True)
    agree = all(all((res[i][k] == res[0][k]).all() for k in range(3)) for i in (1, 2))
    ok = None if (args.fast_setup or args.no_verify) else _verify_proof(syn, res[0])
    if not agree or ok is False:
        raise SystemExit("bench rep3 (1 GPU): proof invalid or parties disagree")
    run(max(1, args.warmup - 1), True)
    sent0 = nets0[0].bytes_sent + nets1[0].bytes_sent
    ms_dev, _ = run(args.steps, True)
    sent = (nets0[0].bytes_sent + nets1[0].bytes_sent - sent0) // args.steps
    ms_host, _ = run(args.steps, False)
    out = {"layout": "3 parties as 3 host threads sharing 1xB200 (one context, key and stream set per party)",
           "gpus": 1, "groups": 1, "gpus_per_party": "1/3",
           "ms_per_proof": ms_dev / args.steps, "proofs_per_s": args.steps / (ms_dev * 1e-3),
           "e2e_ms_per_proof": ms_host / args.steps, "e2e_proofs_per_s": args.steps / (ms_host * 1e-3),
           "h2d_bytes_per_party_per_proof": int(host_sh[0][0].nbytes + pub.nbytes),
           "net_bytes_per_party_per_proof": int(sent), "parties_agree": bool(agree), "pairing_verified": ok,
           "transport": "mailboxes in HBM, in-process (cs_net_peer_connect_local)", "protocol": "cs_groth16_rep3_prove (C++, in-library)",
           "extra_key_upload_s": round(key_s, 2)}
    for i in range(3):
        ctxs[i].free(dev_sh[i])
        nets0[i].free()
        nets1[i].free()
        states[i].free()
    for p_, c_ in zip(pks[1:], ctxs[1:]):
        p_.free()
        c_.close()
    return out


def plonk_rep3_block(args, rank, local_rank):
    """Rep3 co-Plonk (BASELINE configs[3]: domain 2^22, 3 parties on 3 GPUs) on ranks 0-2 of the running job: products
    stored into the next party's GPU over NVLink by the kernels, the party driver inside the library (cs_plonk_rep3_prove),
    proof checked by the oracle's verifier on rank 0.  Every rank calls this (new_group is collective)."""
    import torch.distributed as dist
    group = dist.new_group([0, 1, 2])
    if rank > 2:
        return None
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import time_co_plonk as T
    lg = args.plonk_log_n
    try:
        res = T.measure_group(group, local_rank, [lg], reps=3)
    except Exception as e:  # noqa: BLE001  -- the Groth16 line must still be printed
        return {"error": "%s: %s" % (type(e).__name__, e)} if rank == 0 else None
    if res is None:
        return None
    r = res["2p%d" % lg]
    return {"workload": "co-Plonk Rep3, BN254, synthetic snarkjs-style circuit, domain 2^%d, 3 parties on 3xB200 "
                        "(BASELINE.json configs[3])" % lg,
            "ms_per_proof": r["ms_per_proof"], "proofs_per_s": r["proofs_per_s"], "pairing_verified": r["verified"],
            "net_bytes_per_party_per_proof": r["bytes_sent_per_party"], "key_setup_s": r["setup_s"],
            "timing": "wall clock per proof from host share buffers to the opened proof, max over the three ranks, "
                      "mean of 2 proofs after 1 warm-up",
            "driver": r.get("driver"),
            "transport": "CUDA-IPC mailboxes for tokens / points; products stored into the next party's HBM by the kernels, "
                         "n-sized openings read from the peers' HBM (NVLink)"}


def rep3_multi_gpu(args, ctx, pk, syn, groups, gpp, rank, world, local_rank):
    """One Rep3 proving group per entry of `groups` (global ranks, party-major: [p0 main, (p0 helper), p1 main, ...]);
    one process per GPU, party exchange through CUDA-IPC mailboxes in peer HBM (NVLink), protocol in the library.
    Every rank of the world calls this (ranks outside all groups only take part in the collectives)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from co_snarks_b200 import binding as B
    lib = ctx.lib
    mine = None
    for g, mem in enumerate(groups):
        if rank in mem:
            k = mem.index(rank)
            mine = (g, k // gpp, k % gpp)  # group, party, role (0 = protocol GPU, 1 = helper)
    net0 = net1 = pair = None
    z64 = np.zeros(64, dtype=np.uint8)
    if mine:
        _, pid, role = mine
        if role == 0:
            net0, net1 = B.Net.peer(ctx, pid, 3), B.Net.peer(ctx, pid, 3)
        if gpp == 2:
            pair = B.Net.peer(ctx, role, 2)
    # bootstrap: every rank publishes its three handles (zeros where it has none)
    hs = np.stack([net0.handle() if net0 else z64, net1.handle() if net1 else z64, pair.handle() if pair else z64])
    t = torch.from_numpy(hs.copy()).cuda()
    allh = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(allh, t)
    allh = [x.cpu().numpy() for x in allh]
    if mine:
        g, pid, role = mine
        mem = groups[g]
        if role == 0:
            mains = [mem[p * gpp] for p in range(3)]
            net0.connect(np.stack([allh[r][0] for r in mains]))
            net1.connect(np.stack([allh[r][1] for r in mains]))
        if gpp == 2:
            pr = [mem[pid * 2], mem[pid * 2 + 1]]
            pair.connect(np.stack([allh[r][2] for r in pr]))
    torch.cuda.synchronize()
    dist.barrier()
    state = None
    res = None
    pub = syn.public_inputs
    host_sh = dev_sh = None
    if mine:
        g, pid, role = mine
        xs = _rep3_shares(ctx, syn, B.CS_BN254)
        host_sh = _party_shares(xs, pid)
        dev_sh = ctx.to_device(host_sh[0])
        if role == 0:
            state = B.Rep3StateC.create(net0)  # OS entropy, seeds exchanged over the mailboxes (Rep3State::new)
            if gpp == 2:  # the helper GPU mirrors the party's streams
                s1, p1, s2, p2, _ = state.prf()
                pair.send(1, s1 + s2 + int(p1).to_bytes(8, "little") + int(p2).to_bytes(8, "little"))
        else:
            b = pair.recv(0, 80)
            state = B.Rep3StateC.from_seeds(lib, pid, b[:32], b[32:64], int.from_bytes(b[64:72], "little"),
                                            int.from_bytes(b[72:80], "little"))

    def one(device):
        if not mine:
            return None
        _, pid, role = mine
        hw = None if device else host_sh[0]
        dw = dev_sh if device else None
        if role == 1:
            pk.rep3_prove_helper(pid, pair, state, pub, hw, dw)
            return None
        return pk.rep3_prove(net0, net1, state, pub, hw, dw, pair=pair)

    def timed(steps, device):
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = None
        for _ in range(steps):
            r = one(device)
        torch.cuda.synchronize()
        dt = torch.tensor([(time.perf_counter() - t0) * 1e3 if mine else 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return float(dt.item()), r
    _, res = timed(1, True)
    # agreement: all protocol ranks of a group hold the same opened proof
    flat = np.concatenate([x.reshape(-1) for x in res]) if res is not None else np.zeros(32, dtype=np.uint64)
    tt = torch.from_numpy(flat.view(np.int64).copy()).cuda()
    outs = [torch.empty_like(tt) for _ in range(world)]
    dist.all_gather(outs, tt)
    agree = True
    for mem in groups:
        mains = [mem[p * gpp] for p in range(3)]
        agree = agree and all(bool((outs[r] == outs[mains[0]]).all()) for r in mains)
    ok = None
    if rank == 0 and not (args.fast_setup or args.no_verify):
        ok = _verify_proof(syn, res)
        if not ok or not agree:
            raise SystemExit("bench rep3: proof invalid or parties disagree")
    timed(max(1, args.warmup - 1), True)
    sent0 = (net0.bytes_sent + net1.bytes_sent) if net0 else 0
    ms_dev, _ = timed(args.steps, True)
    sent = ((net0.bytes_sent + net1.bytes_sent - sent0) // args.steps) if net0 else 0
    ms_host, _ = timed(args.steps, False)
    ng = len(groups)
    out = {"layout": "%d group(s) of 3 parties x %d GPU(s) per party, one process per GPU" % (ng, gpp),
           "gpus": ng * 3 * gpp, "groups": ng, "gpus_per_party": gpp,
           "ms_per_proof": ms_dev / args.steps, "proofs_per_s": ng * args.steps / (ms_dev * 1e-3),
           "e2e_ms_per_proof": ms_host / args.steps, "e2e_proofs_per_s": ng * args.steps / (ms_host * 1e-3),
           "h2d_bytes_per_party_per_proof": int((host_sh[0].nbytes if host_sh else 0) + pub.nbytes) * gpp,
           "net_bytes_per_party_per_proof": int(sent), "parties_agree": bool(agree), "pairing_verified": ok,
           "transport": "CUDA-IPC mailboxes in peer HBM (NVLink peer copies), 4 point-sized messages per party",
           "protocol": "cs_groth16_rep3_prove (C++, in-library)"}
    dist.barrier()
    if mine:
        ctx.free(dev_sh)
        for n_ in (net0, net1, pair):
            if n_:
                n_.free()
        state.free()
    return out


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from co_snarks_b200 import binding as B
    from workloads.synth_groth16 import SynthGroth16, BN254_R

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream()
    ctx = B.Context(local_rank, stream=stream.cuda_stream)
    lg = args.log_m
    n = 1 << lg

    # ---- workload (untimed): valid synthetic key with known toxic waste, uploaded once
    t0 = time.time()
    syn = SynthGroth16(ctx, lg, seed=1, setup_seed=2, valid=not args.fast_setup)
    t1 = time.time()
    pk = syn.make_key(args.window_bits)  # cs_groth16_pk_create: matrices + five query arrays -> resident tables
    ctx.synchronize()
    key_upload_s = time.time() - t1
    setup_s = time.time() - t0
    rng = np.random.Generator(np.random.PCG64(3))
    rs = B.ints_to_limbs(B.to_mont_ints([int(rng.integers(1, 2 ** 62)) * 0x10001 % BN254_R for _ in range(2)], BN254_R, 4), 4)
    r_m, s_m = rs[0:1].copy(), rs[1:2].copy()
    pub = syn.public_inputs
    wit_np = syn.private_witness
    wit_pinned = torch.empty(wit_np.shape, dtype=torch.int64).pin_memory()
    wit_pinned.numpy().view(np.uint64)[:] = wit_np
    wit_host = wit_pinned.numpy().view(np.uint64)
    d_wit = ctx.to_device(wit_np)
    h2d = wit_np.nbytes + pub.nbytes
    d2h = 5 * 4 * 8 * 8 + 8 * 8  # five XYZZ results (G2: 2x) land in pinned memory; upper bound, tiny

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- correctness gate before timing: the proof must verify (pairing check, oracle verifier)
    proof_ok = None
    if rank == 0 and not args.fast_setup and not args.no_verify:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from helpers import Conv
        from oracle.pairing_bn254 import groth16_verify
        cv = Conv("bn254")
        A, Bp, Cp = pk.prove_plain(pub, wit_host, r_m, s_m)
        proof_ok = bool(groth16_verify(syn.vk_ints(), syn.witness[1:2], (cv.pt1(A), cv.pt2(Bp), cv.pt1(Cp))))
        if not proof_ok:
            raise SystemExit("bench: proof does not verify -- refusing to time an incorrect path")

    # ---- warm-up
    for _ in range(args.warmup):
        pk.prove_plain(pub, wit_host, r_m, s_m)
        pk.prove_plain_device(pub, d_wit, r_m, s_m)

    # ---- value: device-resident witness, CUDA events on the launching stream
    barrier()
    clocks = ClockSampler(local_rank)
    l0 = ctx.launch_count()
    with torch.cuda.stream(stream):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        tw0 = time.perf_counter()
        for _ in range(args.steps):
            proof = pk.prove_plain_device(pub, d_wit, r_m, s_m)
        e1.record(stream)
    torch.cuda.synchronize()
    tw1 = time.perf_counter()
    dev_ms = max(e0.elapsed_time(e1), 0.0)
    # the proof ends with a short host tail after the last kernel; charge the larger of the two clocks
    value_ms = max_over_ranks(max(dev_ms, (tw1 - tw0) * 1e3))
    launches = ctx.launch_count() - l0
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("proof_a", "proof_b", "proof_c"), proof)))

    timeline = None
    if args.timeline and rank == 0:
        ctx.msm_profile(True)
        tls = []
        for _ in range(3):
            pk.prove_plain_device(pub, d_wit, r_m, s_m)
            tls.append(ctx.msm_timeline_ms())
        ctx.msm_profile(False)
        names = ["A", "B1", "B2", "L", "H"]
        timeline = {"order": "ms after the fork: start, digits done, sort done, accumulate done, fold done, reduce done",
                    "stream_prio": os.environ.get("CS_STREAM_PRIO", "")}
        for w, nm in enumerate(names):
            timeline[nm] = [round(x, 3) for x in tls[-1][w]]
        print("timeline", json.dumps(timeline), file=sys.stderr, flush=True)

    # ---- e2e: host buffers through the C ABI, wall clock between synchronisations
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pk.prove_plain(pub, wit_host, r_m, s_m)
    torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    clk = clocks.stop()
    barrier()
    # the same call from PAGEABLE host memory (what a Rust Vec<Fr> is), first call after an idle period included
    wit_pageable = np.array(wit_np, copy=True)
    t0 = time.perf_counter()
    pk.prove_plain(pub, wit_pageable, r_m, s_m)
    torch.cuda.synchronize()
    pageable_first_ms = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    for _ in range(3):
        pk.prove_plain(pub, wit_pageable, r_m, s_m)
    torch.cuda.synchronize()
    pageable_ms = (time.perf_counter() - t0) * 1e3 / 3
    barrier()

    # ---- the metric's own configuration in the same run: co-Groth16, 3-party Rep3 (BASELINE configs[2]),
    # whole protocol inside the library.  N = 1: three party threads share the GPU; N >= 3: one party per GPU
    # (N // 3 proving groups); N >= 6 additionally 3 parties x 2 GPUs.
    rep3 = rep3_split = None
    if not args.no_rep3:
        if world == 1:
            rep3 = rep3_threads_one_gpu(args, ctx, pk, syn)
        elif world >= 3:
            groups = [[3 * g, 3 * g + 1, 3 * g + 2] for g in range(world // 3)]
            rep3 = rep3_multi_gpu(args, ctx, pk, syn, groups, 1, rank, world, local_rank)
            if world >= 6:
                rep3_split = rep3_multi_gpu(args, ctx, pk, syn, [list(range(6))], 2, rank, world, local_rank)
        barrier()

    # ---- BASELINE configs[3] in the same run when three GPUs are there: Rep3 co-Plonk at domain 2^22 on ranks 0-2
    plonk_blk = None
    if world >= 3 and not args.no_rep3 and not args.no_plonk:
        plonk_blk = plonk_rep3_block(args, rank, local_rank)
        barrier()

    out = None
    if rank == 0:
        # ---- kernel roofline (rank 0, single stream): standalone G1 MSM over a_query with stage events
        hbm, hbm_src = peaks()
        ctx.msm_profile(True)
        # h_query is dense (no points at infinity) and gets uniform 254-bit scalars: the clean MSM case
        nw = n
        a_bases = ctx.bases_upload(B.CS_BN254, B.CS_G1, syn.points["h_query"], args.window_bits)
        d_hs = ctx.to_device(np.resize(wit_np, (n, 4)))
        stage = np.zeros(5)
        msm_ms = []
        reps = max(3, args.steps)
        for i in range(2 + reps):
            with torch.cuda.stream(stream):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                ctx.msm(a_bases, d_hs, offset=0, n=nw, montgomery=True, device=True)
                e1.record(stream)
            torch.cuda.synchronize()
            if i >= 2:
                stage += np.array(ctx.msm_stage_ms())
                msm_ms.append(e0.elapsed_time(e1))
        stage /= reps
        ctx.msm_profile(False)
        a_bases.free()
        ctx.free(d_hs)
        msm_avg = sum(msm_ms) / len(msm_ms)
        accum_ms = float(stage[2])
        alg_bytes = 96.0 * nw  # SURVEY 8(d): 64 B base + 32 B scalar per pair (G1 BN254)
        achieved = alg_bytes / (accum_ms * 1e-3) / 1e9
        # NTT 2^20 (one inverse + one forward over a resident vector)
        dom = ctx.domain(B.CS_BN254, lg, ctx.roots_of_unity(B.CS_BN254, lg)[0])
        d_v = ctx.to_device(np.resize(wit_np, (n, 4)))
        ntt_ms = []
        for i in range(2 + reps):
            with torch.cuda.stream(stream):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                dom.ifft_in_to_out(d_v, 1)
                dom.fft_out_to_in(d_v, 1)
                e1.record(stream)
            torch.cuda.synchronize()
            if i >= 2:
                ntt_ms.append(e0.elapsed_time(e1) / 2)
        ntt_avg = sum(ntt_ms) / len(ntt_ms)
        ctx.free(d_v)
        dom.free()
        gmul_peak, imad_tops, peak_src = int_pipe_ceiling()
        g1_madds = 16.0 * nw  # W = 16 windows: one mixed addition (8M + 2S = 10 products) per scalar per window
        gmul = g1_madds * 10 / (accum_ms * 1e-3) / 1e9
        steps_total = args.steps * world
        out = {
            "metric": METRIC, "value": steps_total / (value_ms * 1e-3), "unit": "proofs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": value_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32x8 (256-bit Montgomery, integer)",
            "data": "synthetic (seeded R1CS + known-toxic-waste key; proof pairing-verified: %s)" % proof_ok,
            "config": {"workload": "plain Groth16 prover, BN254, synthetic R1CS 2^%d constraints, 1xB200 per replica "
                                   "(BASELINE.json configs[1])" % lg,
                       "domain": n, "window_bits": pk_window(args, n), "replicas": world,
                       "l2": "working set (5 precomputed base tables, ~6.4 GB) exceeds the 126 MB L2; no flush needed",
                       "setup_s": round(setup_s, 1), "key_upload_s": round(key_upload_s, 2),
                       "time_to_first_proof_note": "key_upload_s = cs_groth16_pk_create alone (CSR + 5 query arrays uploaded and "
                                                   "expanded to per-window tables); setup_s adds the synthesis of the synthetic key"},
            "e2e": {"value": steps_total / (e2e_ms * 1e-3), "unit": "proofs/s", "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "pageable_host_memory_ms_per_step": pageable_ms, "pageable_first_call_ms": pageable_first_ms},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": {"kernel": "k_msm_accum0<Fp<Bn254Fq>> (G1 bucket accumulation)", "bound": "hbm",
                         "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                         "traffic": ncu_traffic(), "peak_source": hbm_src,
                         "traffic_source": "profiles/r2_ncu_full_accum0_g1.csv (ncu --set full of this kernel on a dense 2^20 G1 MSM; "
                                           "bytes per launch). 16 precomputed table points are read per scalar by design (no doublings), "
                                           "HBM stays below 10 % busy",
                         "note": "256-bit modular arithmetic is integer-pipe bound (~2.3 kIMAD per 96 B); see DESIGN.md",
                         "launch_ms": accum_ms, "algorithmic_bytes_per_launch": alg_bytes,
                         "int_pipe": {"achieved_gmodmul_s": gmul, "peak_gmodmul_s": gmul_peak, "frac": gmul / gmul_peak,
                                      "imad_wide_tops": imad_tops, "imad_wide_tops_source": "profiles/r2_pipe_probe.json (data-dependent operands)", "peak_source": peak_src,
                                      "note": "the resource that actually bounds the kernel: 10 Montgomery products per mixed addition, counted as 10 although two of them (R (Q - X3) - Y1 PPP) share one reduction (Fp::dot2, 1.5 product-equivalents of multiply work)"}},
            "msm": {"g1_2p%d_ms" % lg: msm_avg, "mscalar_per_s": nw / (msm_avg * 1e-3) / 1e6,
                    "stage_ms": {"digits": float(stage[0]), "sort": float(stage[1]), "accumulate": float(stage[2]),
                                 "fold": float(stage[3]), "reduce": float(stage[4])}},
            "ntt": {"2p%d_ms" % lg: ntt_avg, "gbs_algorithmic": 64.0 * n / (ntt_avg * 1e-3) / 1e9,
                    "gmodmul_s": n * lg / 2 / (ntt_avg * 1e-3) / 1e9,
                    "int_pipe_frac": n * lg / 2 / (ntt_avg * 1e-3) / 1e9 / gmul_peak,
                    "note": "n/2 log n butterflies of one Montgomery product each: integer-pipe bound like the MSM"},
            "cpu_baseline": cpu_baseline(args) if (world == 1 and not args.no_cpu_baseline) else None,  # rank 0 at N = 1 only
            **({"timeline_ms": timeline} if timeline else {}),
            "rep3": rep3 if rep3 is not None else ("skipped (--no-rep3)" if args.no_rep3 else "needs 1 or >= 3 GPUs"),
        }
        if rep3_split is not None:
            out["rep3_2gpu_per_party"] = rep3_split
        if plonk_blk is not None:
            out["plonk_rep3"] = plonk_blk
    pk.free()
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        print(json.dumps(out))


def dump_outputs(out_dir, arrays):
    """Writes each uint64 limb array as out_dir/<name>.npy: its 32-bit words (little-endian order) as float64, which
    holds them exactly, so two builds can be compared word for word."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        words = np.ascontiguousarray(a, dtype=np.uint64).view(np.uint32).astype(np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), words)


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the accumulate kernel from the committed ncu summary."""
    path = os.path.join(ROOT, "profiles", "r2_ncu_full_accum0_g1.csv")
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        tot = 0.0
        for line in open(path):
            f = line.strip().split(",")
            if f[0] == "0" and f[1] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                tot += float(f[3].strip('"')) * mult[f[2]]
        return tot or None
    except OSError:
        return None


def run_rep3(args):
    """Standalone BASELINE configs[2]: torchrun --nproc-per-node 3 (or 6 with --gpus-per-party 2) bench.py --mode rep3.
    One step = one collaborative proof; the same code path as the `rep3` block of the default run."""
    import torch
    import torch.distributed as dist
    from co_snarks_b200 import binding as B
    from workloads.synth_groth16 import SynthGroth16
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    gpp = args.gpus_per_party
    assert gpp in (1, 2) and world % (3 * gpp) == 0, "rep3 mode needs 3 (or 6) ranks per proving group"
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream()
    ctx = B.Context(local_rank, stream=stream.cuda_stream)
    t0 = time.time()
    syn = SynthGroth16(ctx, args.log_m, seed=1, setup_seed=2, valid=not args.fast_setup)
    pk = syn.make_key(args.window_bits)
    setup_s = time.time() - t0
    blk = 3 * gpp
    groups = [list(range(g * blk, (g + 1) * blk)) for g in range(world // blk)]
    clocks = ClockSampler(local_rank)
    l0 = ctx.launch_count()
    r = rep3_multi_gpu(args, ctx, pk, syn, groups, gpp, rank, world, local_rank)
    launches = ctx.launch_count() - l0
    clk = clocks.stop()
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": r["proofs_per_s"], "unit": "proofs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["ms_per_proof"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32x8 (256-bit Montgomery, integer)",
            "data": "synthetic (seeded R1CS + known-toxic-waste key; proof pairing-verified: %s; parties agree: %s)" % (
                r["pairing_verified"], r["parties_agree"]),
            "config": {"workload": "co-Groth16 Rep3, BN254, synthetic R1CS 2^%d constraints, 3 parties x %d GPU(s), "
                                   "(BASELINE.json configs[2])" % (args.log_m, gpp), "setup_s": round(setup_s, 1),
                       "l2": "working set exceeds L2"},
            "e2e": {"value": r["e2e_proofs_per_s"], "unit": "proofs/s", "h2d_bytes_per_step": r["h2d_bytes_per_party_per_proof"],
                    "d2h_bytes_per_step": 1344},
            "gpu_launches": int(launches), "clocks": clk, "rep3": r}))
    pk.free()
    ctx.close()
    dist.barrier()
    dist.destroy_process_group()


def run_plonk_rep3(args):
    """BASELINE.json configs[3]: co-Plonk Rep3, BN254, synthetic circuit of domain 2^log_m, 3 parties on 3 GPUs.
    torchrun --nproc-per-node 3 bench.py --mode plonk-rep3 --log-m 22.  One step = one collaborative proof
    (first-layer products stored into the next party's GPU over NVLink peer memory, openings over NCCL)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import time_co_plonk as T
    res = T.measure([args.log_m], reps=args.steps + 1)
    if res is None:
        return
    r = res["2p%d" % args.log_m]
    print(json.dumps({
        "metric": "co-Plonk Rep3 proofs/sec (BN254, domain 2^%d)" % args.log_m, "value": r["proofs_per_s"], "unit": "proofs/s",
        "n_gpus": 3, "steps": args.steps, "warmup": 1, "ms_per_step": r["ms_per_proof"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32x8 (256-bit Montgomery, integer)",
        "data": "synthetic snarkjs-style Plonk circuit with a valid key; proof accepted by the oracle's verifier: %s" % r["verified"],
        "config": {"workload": "co-Plonk Rep3, BN254, synthetic circuit domain size 2^%d, 3 parties on 3xB200 "
                               "(BASELINE.json configs[3])" % args.log_m, "setup_s": r["setup_s"]},
        "e2e": {"value": r["proofs_per_s"], "unit": "proofs/s", "note": "host share buffers in, opened proof out, wall clock, max over ranks"},
        "net_bytes_per_party_per_proof": r["bytes_sent_per_party"]}))


def int_pipe_ceiling():
    """Measured ceiling of 256-bit Montgomery products on the integer pipe (tools/imad_peak, built by
    __graft_entry__.build()); falls back to the committed measurement of this pool's B200."""
    exe = os.path.join(ROOT, "tools", "imad_peak")
    try:
        out = subprocess.run([exe], capture_output=True, text=True, timeout=120).stdout
        j = json.loads(out)
        # the probe's own "imad_wide_tops" loop has loop-invariant operands that ptxas strength-reduces to adds (it reads
        # 17 T/s); the IMAD.WIDE issue rate with data-dependent operands is 9.2 T/s (tools/pipe_probe.cu,
        # profiles/r2_pipe_probe.json), which is what the Montgomery ceiling below reflects
        return max(v for k, v in j.items() if k.startswith("montmul_gmuls")), 9.2, "measured live (tools/imad_peak)"
    except Exception:  # noqa: BLE001
        return 65.2, 9.2, "committed measurement (profiles/r1_imad_peak_and_multiplier_variants.json)"


def pk_window(args, n):
    return args.window_bits or 16


def cpu_baseline(args):
    """The oracle's C restatement timed on the host cores on a bounded sample (rank 0, N = 1 only)."""
    try:
        from oracle.c import run as oc
    except Exception as e:  # noqa: BLE001
        return {"value": None, "unit": "proofs/s", "cores": 0, "kind": "port", "sample": "unavailable: %s" % e}
    return oc.cpu_baseline(log_m=args.cpu_log_m, target_log_m=args.log_m)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.c import run as oc
    res = oc.reference_arm(log_m=args.cpu_log_m, target_log_m=args.log_m, steps=args.steps, warmup=args.warmup)
    res["n_gpus"] = args.gpus  # the launch it mirrors (the arm itself runs on host cores only, rank 0)
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-m", type=int, default=20, help="log2 of the number of R1CS variables / domain size")
    ap.add_argument("--cpu-log-m", type=int, default=20, help="log2 size of the CPU baseline sample")
    ap.add_argument("--window-bits", type=int, default=0)
    ap.add_argument("--mode", default="plain", choices=["plain", "rep3", "plonk-rep3"])
    ap.add_argument("--gpus-per-party", type=int, default=1)
    ap.add_argument("--fast-setup", action="store_true", help="random (invalid) key: skips the host-side QAP setup")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-rep3", action="store_true", help="skip the Rep3 block of the default run")
    ap.add_argument("--no-plonk", action="store_true", help="skip the co-Plonk block of runs with >= 3 GPUs")
    ap.add_argument("--plonk-log-n", type=int, default=22, help="log2 domain size of the co-Plonk block")
    ap.add_argument("--timeline", action="store_true",
                    help="after the timed region: one more proof with stage events, reported as timeline_ms (diagnostic)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="diagnostic runs: skip the CPU leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the proof (A, B, C) of the last timed step as DIR/proof_{a,b,c}.npy: the affine Montgomery "
                         "limbs the prover returns, as float64 32-bit words")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.mode == "rep3":
        run_rep3(args)
    elif args.mode == "plonk-rep3":
        run_plonk_rep3(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
