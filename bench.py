#!/usr/bin/env python
"""bench.py -- headline benchmark: BLS aggregate-verify sigs/s on the 250-validator FBFT commit batch (BASELINE.json).

A "step" = one pass of the hot path over one batch of synthetic input: B independent commit rounds
(bitmap32 || aggSig96 || payload48 each, BASELINE configs[1]) verified against one device-resident 250-key
committee, i.e. B x { Mask.SetMask ; Sign.Deserialize ; aggSig.VerifyHash(mask.AggregatePublic, payload) }
(reference internal/chain/engine.go:619-642).  `value` counts constituent signatures (set bits) per second with the
inputs already in HBM; `e2e` is the same metric through the host-buffer C-ABI call (H2D/D2H inside the timed region).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--rounds B] [--impl reference] [--dump-outputs DIR]
Multi-GPU: torchrun, one rank per GPU; rounds shard by index with no data-path collective (weak scaling).
--dump-outputs DIR writes the per-round results of the last timed step as DIR/aggregate_verify_results.npy (float32, 1 = the
round verifies); the inputs are seeded, so two builds can be compared output for output.
"""
import argparse, ctypes, json, os, subprocess, sys, threading, time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it (it may be read-only)
sys.path.insert(0, ROOT)
import numpy as np
from harmony_b200 import workload as wl

N_COMMITTEE = 250
MSG_LEN = 48
MAC32_PER_MUL, MAC32_PER_SQR = 300, 234          # SURVEY.md 8d fixed conversion (12-limb CIOS)

def log(*a):
    print(*a, file=sys.stderr, flush=True)

# ------------------------------------------------------------------ synthetic workload (deterministic, byte-level only)
def make_committee_sks(n=N_COMMITTEE):
    return [wl.seeded_sk("c2", i) for i in range(n)]

def make_rounds(sks, B, seed, rank=0):
    """B rounds: distinct bitmap (k cycles 167/200/250 = quorum .. full), distinct 48-byte commit payload,
    and the secret scalar sum(sk_i over the bitmap) mod r whose SignHash IS the round's aggregate signature."""
    n = len(sks)
    rng = np.random.Generator(np.random.Philox(key=[seed, rank]))
    ks = np.array([wl.quorum_k(n), 200, n], dtype=np.int64)[np.arange(B) % 3]
    order = np.argsort(rng.random((B, n)), axis=1)
    member = np.zeros((B, n), dtype=bool)
    np.put_along_axis(member, order, np.arange(n)[None, :] < ks[:, None], axis=1)
    padded = np.zeros((B, ((n + 7) // 8) * 8), dtype=np.uint8); padded[:, :n] = member
    bitmaps = np.packbits(padded, axis=1, bitorder="little")                       # LSB-first (mask.go:110-112)
    limbs = np.array([[(k >> (32 * j)) & 0xffffffff for j in range(8)] for k in sks], dtype=np.int64)
    sums = member.astype(np.int64) @ limbs                                          # B x 8, each < 250 * 2^32
    agg_sk = b"".join(wl.sk_bytes(sum(int(sums[b, j]) << (32 * j) for j in range(8))) for b in range(B))
    payload = np.zeros((B, MSG_LEN), dtype=np.uint8)                                # LE64(blockNum) || hash32 || LE64(viewID)
    payload[:, 0:4] = rng.integers(0, 256, (B, 4), dtype=np.uint8)
    payload[:, 8:40] = rng.integers(0, 256, (B, 32), dtype=np.uint8)
    payload[:, 40:44] = rng.integers(0, 256, (B, 4), dtype=np.uint8)
    nsig = int(member.sum())
    return bitmaps.tobytes(), agg_sk, payload.tobytes(), nsig

# ------------------------------------------------------------------ clocks
class ClockSampler:
    def __init__(self, dev):
        self.dev = dev; self.samples = []; self.reasons = set(); self.stop = False; self.t = None; self.maxmhz = None
    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.dev), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0])); self.maxmhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v: self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.1)
    def start(self): self.t = threading.Thread(target=self._run, daemon=True); self.t.start()
    def finish(self):
        self.stop = True
        if self.t: self.t.join(timeout=6)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.maxmhz, "reasons": sorted(self.reasons), "samples": len(s)}

# ------------------------------------------------------------------ CPU arm (oracle = restated reference path; see DESIGN.md)
def usable_cores():
    """Host threads this process may actually use: sched affinity, capped by the cgroup CPU quota (cpu.max / cfs_quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max": quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0: quota = q / per
        except Exception: pass
    info = {"affinity": n, "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}
    if quota: n = max(1, min(n, int(quota + 0.5)))
    return n, info

def oracle_lib():
    """The only place bench.py touches oracle/: cpu_baseline leg and --impl reference."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    return ol.load()

def cpu_rounds_per_s(orc, pks, bitmaps, sigs, msgs, blen, budget_s, threads):
    """Reference call pattern per round: NewMask+SetMask (250 G1 adds) ; Sign.Deserialize ; VerifyHash, on `threads` host threads
    (ctypes releases the GIL).  Runs ~budget_s seconds; returns (rounds/s, rounds done, all results correct)."""
    B = len(sigs) // 96
    h = orc.committee(pks)
    done = [0] * threads; good = [True] * threads
    t_end = time.perf_counter() + budget_s
    def work(t):
        j = t
        while time.perf_counter() < t_end:
            r = j % B
            rc = orc.committee_aggregate_verify(h, bitmaps[r * blen:(r + 1) * blen], sigs[r * 96:(r + 1) * 96], msgs[r * MSG_LEN:(r + 1) * MSG_LEN])
            good[t] &= (rc == 1); done[t] += 1; j += threads
    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    [t.start() for t in ths]; [t.join() for t in ths]
    dt = time.perf_counter() - t0
    return sum(done) / dt, sum(done), all(good)

# EXECUTED work per round = Fp multiplications / squarings the device code performs, counted by running the very same kernels on
# the host (tests/emu/emu_kernels.cpp: emu_stage_counts for the thread-per-item stages, tests/emu/emu_main.cpp: emu_rlc_stage_counts
# for the lane-pair pairing stage); pinned by tests/test_emu_kernels.py::test_stage_counts_pinned and tests/test_emu_logic.py.
# (mul, sqr); "scale"/"pairing" are per GROUP of G rounds, the others per round of the 167/200/250-signer workload.
EXEC_FP_OPS = {
    False: {"mask": (368.5, 137.8), "decode": (1478.0, 756.0), "hash": (3173.4, 1524.0),
            4: {"scale": (4927.0, 2587.0), "pairing": (32456, 764)}, 8: {"scale": (11255.0, 5032.0), "pairing": (50360, 764)}},
    True: {"mask": (368.5, 137.8), "decode": (1478.0, 756.0), "hash": (3004.2, 855.5),
            4: {"scale": (4571.5, 1257.0), "pairing": (32456, 764)}, 8: {"scale": (10544.0, 2372.0), "pairing": (50360, 764)}},      # shared inversions (HB_BATCH_INV, 8 items per inversion)
}
EXEC_FP_OPS_LINES = {4: (8900, 0), 8: (16020, 0)}     # the line kernel's share of "pairing" in the two-kernel form (k_rlc_lines_split; tests/test_emu_logic.py)
EXACT_PAIRING_FP_OPS = (20055, 497)      # exact mode: 2-pair Miller loop + final exponentiation per round (oracle counter, stages 4 + 5)
def rlc_group_size(B, sm_count, tpb_split=512):
    """Mirror of the host's choice in hbls.cu launch_verify_tail: 8 when B/8 lane pairs still fill every SM, else 4."""
    env = os.environ.get("HBLS_RLC_G")
    if env in ("4", "8"): return int(env)
    return 8 if 2 * (B // 8) >= sm_count * tpb_split else 4
def mac32(ops): return ops[0] * MAC32_PER_MUL + ops[1] * MAC32_PER_SQR
def executed_mac32_per_round(batch_inv, G):
    t = EXEC_FP_OPS[bool(batch_inv)]
    return [mac32(t["mask"]), 0.0, mac32(t["decode"]), mac32(t["hash"]), mac32(t[G]["scale"]) / G, mac32(t[G]["pairing"]) / G]
def ncu_dram_bytes(kernel_substr):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, read from the newest committed ncu summary
    (profiles/r*_ncu_*.txt written by tools/ncu_summary.py) whose title names that kernel; None if there is none."""
    import glob, re
    best = None
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_*.txt"))):
        try: txt = open(f).read()
        except OSError: continue
        if kernel_substr not in txt.splitlines()[0]: continue
        vals = {}
        for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            m = re.search(r"^" + re.escape(key) + r"\s+([0-9.]+)\s+(\w+)", txt, re.M)
            if m: vals[key] = float(m.group(1)) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}.get(m.group(2), 1)
        if len(vals) == 2: best = (sum(vals.values()), os.path.relpath(f, ROOT))
    return best

def stage_mac32_per_round(orc, pks, bitmaps, sigs, msgs, blen, sample=12):
    """ALGORITHMIC work per round and per pipeline stage from the oracle's Fp mul/sqr counter (SURVEY 8d)."""
    h = orc.committee(pks)
    fn = orc.L.ho_profile_aggregate_verify
    fn.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_uint64)]
    acc = np.zeros(12)
    for r in range(sample):
        out = (ctypes.c_uint64 * 12)()
        rc = fn(h, bitmaps[r * blen:(r + 1) * blen], blen, sigs[r * 96:(r + 1) * 96], msgs[r * MSG_LEN:(r + 1) * MSG_LEN], MSG_LEN, out)
        assert rc == 1
        acc += np.array(list(out), dtype=np.float64)
    acc /= sample
    return [float(acc[2 * s] * MAC32_PER_MUL + acc[2 * s + 1] * MAC32_PER_SQR) for s in range(6)]

# ------------------------------------------------------------------ the other BASELINE configs (C3 / C4 / C5), short legs reported beside the headline
def _median_ms(fn, reps=3):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); out = fn(); ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), out

def other_configs(bls, world, rank, dist, device):
    """C3: 4 shards x 250 validators, 4 distinct messages, one call (+ a 1 024-item multi-committee batch);
    C4: 10 000 independent triples, 1 % invalid -- one GPU through hbls_verify_batch, and split over the ranks (partial records,
        NCCL all-gather, fold; exact per-slice pass when the fold does not settle it);
    C5: 1 000-validator committee: sign 1 000, aggregate 1 000, aggregate-verify at 64 / 256 / 1 024 rounds.
    Host-buffer calls, wall-clock medians (these legs are latency-like: copies and launches included)."""
    from harmony_b200 import shard
    out = {}
    rng = np.random.Generator(np.random.Philox(key=[31337, 0]))
    if rank == 0:
        # ---- C3
        n = N_COMMITTEE; coms, skss = [], []
        for sh in range(4):
            sks = [wl.seeded_sk(f"bench-c3/{sh}", i) for i in range(n)]
            blob = bls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
            coms.append(bls.Committee([blob[48 * i:48 * i + 48] for i in range(n)])); skss.append(sks)
        def items(K):
            idx = [j % 4 for j in range(K)]
            bms = [wl.bitmap_with_k("bench-c3/bm", j, n, [167, 200, 250, 180][j % 4]) for j in range(K)]
            msgs = b"".join(wl.commit_payload("bench-c3/m", j) for j in range(K))
            agg = b"".join(wl.sk_bytes(wl.round_signer_sum(skss[idx[j]], bms[j])) for j in range(K))
            sigs, ok = bls.SignHashBatch(agg, msgs, MSG_LEN)
            return [coms[i] for i in idx], bms, sigs, msgs, sum(sum(bin(b).count("1") for b in bm) for bm in bms)
        for K in (4, 1024):
            cs, bms, sigs, msgs, nsig = items(K)
            ms, res = _median_ms(lambda: bls.AggregateVerifyItems(cs, bms, sigs, msgs, MSG_LEN), 5 if K == 4 else 3)
            assert res == b"\x01" * K
            out[f"c3_items_{K}"] = {"ms": ms, "sigs_per_s": nsig / (ms * 1e-3), "committees": 4, "mode": bls.LastBatchInfo()["mode"]}
        # ---- C5
        n5 = 1000
        sks5 = [wl.seeded_sk("bench-c5", i) for i in range(n5)]
        sk_blob = b"".join(wl.sk_bytes(k) for k in sks5)
        ms_pk, pk_blob = _median_ms(lambda: bls.GetPublicKeyBatch(sk_blob), 1)
        com5 = bls.Committee([pk_blob[48 * i:48 * i + 48] for i in range(n5)])
        m5 = wl.commit_payload("bench-c5", 0)
        ms_sign, (sigs5, ok5) = _median_ms(lambda: bls.SignHashBatch(sk_blob, m5 * n5, MSG_LEN))
        ms_agg, agg5 = _median_ms(lambda: bls.AggregateSigBytes([sigs5[96 * i:96 * i + 96] for i in range(n5)]))
        full_bm = bytes([0xff] * (n5 // 8))
        assert com5.AggregateVerify(full_bm, agg5, m5)
        c5 = {"committee": n5, "sign_1000_ms": ms_sign, "aggregate_1000_sigs_ms": ms_agg, "verify": {}}
        for Bv in (64, 256, 1024):
            bms = [wl.bitmap_with_k("bench-c5/bm", j % 16, n5, [667, 800, 1000][j % 3]) for j in range(Bv)]
            msgs = b"".join(wl.commit_payload("bench-c5/m", j) for j in range(Bv))
            agg = b"".join(wl.sk_bytes(wl.round_signer_sum(sks5, bms[j])) for j in range(Bv))
            sigs, ok = bls.SignHashBatch(agg, msgs, MSG_LEN)
            ms, res = _median_ms(lambda: com5.AggregateVerifyBatch(b"".join(bms), sigs, msgs, MSG_LEN))
            assert res == b"\x01" * Bv
            nsig = sum(sum(bin(b).count("1") for b in bm) for bm in bms)
            c5["verify"][str(Bv)] = {"ms": ms, "sigs_per_s": nsig / (ms * 1e-3)}
        out["c5_super_committee"] = c5
    # ---- C4 (every rank takes part in the split form)
    k = 10000
    sks4 = b"".join(wl.sk_bytes(wl.seeded_sk("bench-c4", i)) for i in range(k))
    msgs4 = b"".join(wl.seeded_bytes("bench-c4/m", i, 32) for i in range(k))
    pks4 = bls.GetPublicKeyBatch(sks4)
    sigs4, ok4 = bls.SignHashBatch(sks4, msgs4, 32)
    bad = np.sort(np.random.Generator(np.random.Philox(key=[4, 4])).choice(k, size=k // 100, replace=False))
    a_sg = np.frombuffer(sigs4, dtype=np.uint8).reshape(k, 96).copy(); a_ms = np.frombuffer(msgs4, dtype=np.uint8).reshape(k, 32).copy()
    a_sg[bad[0::2], 11] ^= 1; a_ms[bad[1::2], 5] ^= 0x80
    sig_bad, msg_bad = a_sg.tobytes(), a_ms.tobytes()
    want = bytearray(b"\x01" * k)
    for i in bad: want[i] = 0
    c4 = {"triples": k, "invalid": int(len(bad))}
    if rank == 0:
        ms, res = _median_ms(lambda: bls.VerifyBatch(pks4, sig_bad, msg_bad, 32))
        assert res == bytes(want)
        c4["one_gpu_verify_batch"] = {"ms": ms, "triples_per_s": k / (ms * 1e-3), "results_exact": True, "batch_info": bls.LastBatchInfo()}
        ms, res = _median_ms(lambda: bls.VerifyBatch(pks4, sigs4, msgs4, 32))
        assert res == b"\x01" * k
        c4["one_gpu_verify_batch_all_valid"] = {"ms": ms, "triples_per_s": k / (ms * 1e-3)}
    if rank == 0:
        # ---- the storm as the reference meets it: one VIEWCHANGE message from every validator of a 250-key committee, 2/3 of them
        # with an embedded PREPARED proof (consensus/view_change_construct.go:237-375 via harmony_b200/consensus.py): two device
        # calls -- 2 n independent triples (messages of 1 / 8 / >= 128 bytes in one 48-byte batch) + the n_m1 quorum proofs
        from harmony_b200 import consensus as cs
        n = N_COMMITTEE; vid = 7
        sksv = [wl.seeded_sk("bench-vc", i) for i in range(n)]
        blobv = bls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sksv)); pksv = [blobv[48 * i:48 * i + 48] for i in range(n)]
        bh = wl.seeded_bytes("bench-vc/hash", 0, 32); bmq = wl.bitmap_with_k("bench-vc/prep", 0, n, wl.quorum_k(n))
        aggp, _ = bls.SignHashBatch(wl.sk_bytes(wl.round_signer_sum(sksv, bmq)), bh, 32)
        payload = bh + aggp + bmq
        is_m1 = [i % 3 != 2 for i in range(n)]
        skb = b"".join(wl.sk_bytes(k) for k in sksv)
        s_vc, _ = bls.SignHashBatch(skb, b"".join(cs._m48(payload if is_m1[i] else cs.NIL) for i in range(n)), 48)
        s_id, _ = bls.SignHashBatch(skb, cs._m48(vid.to_bytes(8, "little")) * n, 48)
        vmsgs = [cs.FBFTMessage(ViewID=vid, BlockNum=1, SenderPubkey=pksv[i], LeaderPubkey=pksv[0], Payload=payload if is_m1[i] else b"",
                                Block=b"\xc0" if is_m1[i] else b"", ViewchangeSig=s_vc[96 * i:96 * i + 96], ViewidSig=s_id[96 * i:96 * i + 96]) for i in range(n)]
        vc = cs.viewChange(pksv)
        def storm():
            vc.Reset(); return vc.ProcessViewChangeMsgs(vmsgs)
        ms, res = _median_ms(storm, 5)
        assert res == [None] * n and not vc.IsM1PayloadEmpty()
        m3sig, m3bm = vc.GetM3Bitmap(vid)
        nv = cs.FBFTMessage(ViewID=vid, BlockNum=1, SenderPubkey=pksv[0], Payload=payload, Block=b"\xc0", M3AggSig=m3sig, M3Bitmap=m3bm)
        nv.M2AggSig, nv.M2Bitmap = vc.GetM2Bitmap(vid)
        ms_nv, err = _median_ms(lambda: vc.OnNewViewChecks(nv), 5)
        assert err is None
        n_m1 = sum(is_m1)
        c4["view_change_handlers"] = {"messages": n, "m1": n_m1, "m2": n - n_m1, "signature_checks": 2 * n + n_m1, "device_calls": 2, "ms": ms,
                                      "messages_per_s": n / (ms * 1e-3), "new_view_checks_ms": ms_nv,
                                      "what": "ProcessViewChangeMsgs over 250 VIEWCHANGE messages (errors and state identical to the sequential reference handlers: tests/test_consensus.py); NEWVIEW = M3 + M2 + M1 aggregate checks in one call"}
    def split(sg, ms_):
        if world > 1: dist.barrier()
        t0 = time.perf_counter()
        res, settled = shard.verify_triples_split(pks4, sg, ms_, 32, device=device)
        dt = (time.perf_counter() - t0) * 1e3
        if world > 1:
            import torch
            t = torch.tensor([dt], dtype=torch.float64, device=device); dist.all_reduce(t, op=dist.ReduceOp.MAX); dt = float(t[0])
        return dt, res, settled
    split(sigs4, msgs4)                                   # warm-up (allocations, NCCL channel set-up)
    v = [split(sigs4, msgs4) for _ in range(3)]
    assert all(r == b"\x01" * k and s for _, r, s in v)
    ms_ok = float(np.median([d for d, _, _ in v]))
    v = [split(sig_bad, msg_bad) for _ in range(3)]
    assert all(r == bytes(want) and not s for _, r, s in v)
    ms_bad = float(np.median([d for d, _, _ in v]))
    c4["split_over_ranks"] = {"ranks": world, "scaling": "strong", "collective": "all-gather of one 872-byte partial record per rank + identical local fold",
                              "all_valid": {"ms": ms_ok, "triples_per_s": k / (ms_ok * 1e-3), "settled_by_fold": True},
                              "one_pct_invalid": {"ms": ms_bad, "triples_per_s": k / (ms_bad * 1e-3), "settled_by_fold": False,
                                                  "note": "fold fails by construction; every rank then verifies its slice exactly and the result bytes are all-gathered"}}
    out["c4_view_change_storm"] = c4
    return out

# ------------------------------------------------------------------ --dump-outputs
DUMP_MAX_BYTES = 64_000_000

def dump_outputs(out_dir, name, results):
    """results (uint8 per round) -> out_dir/<name>.npy as float32.  Beyond DUMP_MAX_BYTES a fixed seeded sample of the rounds is
    written instead, with the sampled round indices beside it in <name>_index.npy (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    res = np.asarray(results, dtype=np.float32)
    if res.nbytes > DUMP_MAX_BYTES:
        keep = DUMP_MAX_BYTES // (4 + 8)
        idx = np.sort(np.random.Generator(np.random.Philox(key=[7, 7])).choice(res.size, size=keep, replace=False))
        np.save(os.path.join(out_dir, name + "_index.npy"), idx.astype(np.float64))
        res = res[idx]
    np.save(os.path.join(out_dir, name + ".npy"), res)

# ------------------------------------------------------------------ main arms
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads, core_info = usable_cores()
    sks = make_committee_sks()
    orc = oracle_lib()
    pks = [orc.get_public_key(wl.sk_bytes(k)) for k in sks]
    S = 64
    bitmaps, agg_sk, msgs, nsig = make_rounds(sks, S, seed=2024)
    sigs = b"".join(orc.sign_hash(agg_sk[32 * j:32 * j + 32], msgs[MSG_LEN * j:MSG_LEN * j + MSG_LEN]) for j in range(S))
    blen = (N_COMMITTEE + 7) // 8
    per = max(1.0, min(8.0, 60.0 / max(1, args.steps + args.warmup)))
    for _ in range(args.warmup):
        cpu_rounds_per_s(orc, pks, bitmaps, sigs, msgs, blen, min(per, 1.0), threads)
    rates = []; ok = True; rounds = 0
    for _ in range(args.steps):
        r, d, g = cpu_rounds_per_s(orc, pks, bitmaps, sigs, msgs, blen, per, threads)
        rates.append(r); ok &= g; rounds += d
    rps = float(np.mean(rates)); sig_per_round = nsig / S
    value = rps * sig_per_round
    rps1, _, _ = cpu_rounds_per_s(orc, pks, bitmaps, sigs, msgs, blen, min(per, 3.0), 1)
    line = {"impl": "reference", "metric": "BLS aggregate-verify sigs/sec (250-validator FBFT commit batch)", "value": value, "unit": "sigs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64 (6x64-bit Montgomery limbs)", "data": "synthetic",
            "config": {"workload": "FBFT commit-phase: 250-validator committee, FastAggregateVerify per round (SetMask + Deserialize + VerifyHash)",
                       "committee": N_COMMITTEE, "msg_len": MSG_LEN, "signers_per_round": "167/200/250 cycling"},
            "cpu_baseline": {"value": value, "unit": "sigs/s", "cores": threads, "kind": "port", "core_info": core_info,
                             "single_thread_value": rps1 * sig_per_round, "thread_scaling": rps / rps1 if rps1 else None,
                             "sample": f"{rounds} rounds over {args.steps} x {per:.1f}s windows on {threads} threads; restated CPU path (oracle/hbls_oracle.c), real libbls not buildable here"},
            "e2e": {"value": value, "unit": "sigs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "all_correct": bool(ok)}
    print(json.dumps(line), flush=True)

def run_gpu(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the BLS backend has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # NCCL's own log (whatever NCCL_DEBUG asks for) goes to stderr: stdout stays one JSON line
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from harmony_b200 import bls
    bls.Init(device=local)
    L = bls.lib()
    B = args.rounds
    blen = (N_COMMITTEE + 7) // 8
    sks = make_committee_sks()
    pks_blob = bls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
    pks = [pks_blob[48 * i:48 * i + 48] for i in range(N_COMMITTEE)]
    com = bls.Committee(pks)
    t0 = time.time()
    bitmaps, agg_sk, msgs, nsig = make_rounds(sks, B, seed=2024, rank=rank)
    sigs, ok = bls.SignHashBatch(agg_sk, msgs, MSG_LEN)
    assert ok == b"\x01" * B
    log(f"[rank {rank}] inputs: {B} rounds, {nsig} constituent sigs, generated in {time.time() - t0:.1f}s")

    # device-resident copies (value) and pinned host copies (e2e)
    def dev(b): return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
    def pin(b): return torch.frombuffer(bytearray(b), dtype=torch.uint8).pin_memory()
    d_bm, d_sig, d_msg = dev(bitmaps), dev(sigs), dev(msgs)
    d_res = torch.zeros(B, dtype=torch.uint8, device="cuda")
    h_bm, h_sig, h_msg = pin(bitmaps), pin(sigs), pin(msgs)
    h_res = torch.zeros(B, dtype=torch.uint8).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")               # > 126 MB L2
    stream = torch.cuda.Stream()

    def step_device():
        rc = L.hbls_aggregate_verify_batch_device(com.h, B, d_bm.data_ptr(), blen, d_sig.data_ptr(), d_msg.data_ptr(), MSG_LEN, d_res.data_ptr(), stream.cuda_stream)
        assert rc == 0, rc
    def step_host():
        rc = L.hbls_aggregate_verify_batch(com.h, B, h_bm.data_ptr(), blen, h_sig.data_ptr(), h_msg.data_ptr(), MSG_LEN, h_res.data_ptr())
        assert rc == 0, rc
    def barrier():
        if world > 1: dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            flush.zero_(); step_device()
    barrier()
    assert int(d_res.sum().item()) == B, "warm-up verification returned a false negative"

    sampler = ClockSampler(local); sampler.start()
    launches0 = bls.KernelLaunchCount()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    stage_ms = np.zeros(6)
    barrier()
    t_wall0 = time.perf_counter()
    with torch.cuda.stream(stream):
        for i in range(args.steps):
            flush.zero_()                                   # L2 flush between timed iterations (outside the event pair)
            evs[i][0].record(stream); step_device(); evs[i][1].record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = bls.KernelLaunchCount() - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    assert int(d_res.sum().item()) == B
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "aggregate_verify_results" + (f"_rank{rank}" if rank else ""), d_res.cpu().numpy())
    # per-kernel durations: separate passes with event records between the kernels (kept out of the timed region)
    bls.StageTimingEnable(True)
    n_stage = 3; lines_ms = 0.0
    with torch.cuda.stream(stream):
        for i in range(n_stage):
            flush.zero_(); step_device()
            st = bls.StageTimingGet(); stage_ms += np.array(st if len(st) == 6 else [0] * 6)
            lines_ms += bls.StageTimingLinesMs()
    bls.StageTimingEnable(False)
    lines_ms /= n_stage
    barrier()
    stage_ms /= n_stage

    def timed_device(n_steps, bm=None, sg=None, ms=None, rounds=None):
        """median CUDA-event time of one device-resident pass over the given (default: the step's) buffers, L2 flushed in between"""
        bm = d_bm if bm is None else bm; sg = d_sig if sg is None else sg; ms = d_msg if ms is None else ms; rounds = B if rounds is None else rounds
        evs2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_steps)]
        with torch.cuda.stream(stream):
            for a_, b_ in [(None, None)] + evs2:          # first pass untimed
                flush.zero_()
                if a_ is not None: a_.record(stream)
                rc = L.hbls_aggregate_verify_batch_device(com.h, rounds, bm.data_ptr(), blen, sg.data_ptr(), ms.data_ptr(), MSG_LEN, d_res.data_ptr(), stream.cuda_stream)
                assert rc == 0, rc
                if b_ is not None: b_.record(stream)
        barrier()
        return float(np.median([a_.elapsed_time(b_) for a_, b_ in evs2]))

    # the exact per-round algorithm (batch mode 0: one 2-pair Miller loop + final exponentiation per round) on the same batch
    bls.SetBatchMode(0)
    exact_ms = timed_device(3)
    assert int(d_res.sum().item()) == B
    bls.SetBatchMode(1)

    # BASELINE C4 rule applied to the headline workload: 1 % of the rounds invalid (wrong payload / signature of another round /
    # flipped participation bit / undecodable signature, seeded positions).  Results must be exactly "all but those"; the rounds of
    # the groups that hold a bad round go through the exact pass (hbls_last_batch_info).
    rng_bad = np.random.Generator(np.random.Philox(key=[99, rank]))
    n_bad = max(1, B // 100)
    bad_idx = np.sort(rng_bad.choice(B, size=n_bad, replace=False))
    a_bm = np.frombuffer(bitmaps, dtype=np.uint8).reshape(B, blen).copy()
    a_sg = np.frombuffer(sigs, dtype=np.uint8).reshape(B, 96).copy()
    a_ms = np.frombuffer(msgs, dtype=np.uint8).reshape(B, MSG_LEN).copy()
    kind = np.arange(n_bad) % 4
    a_ms[bad_idx[kind == 0], 17] ^= 0x20
    src = (bad_idx[kind == 1] + 1) % B; a_sg[bad_idx[kind == 1]] = np.frombuffer(sigs, dtype=np.uint8).reshape(B, 96)[src]
    a_bm[bad_idx[kind == 2], 5] ^= 0x04
    a_sg[bad_idx[kind == 3]] = 0xff
    i_bm, i_sg, i_ms = (torch.from_numpy(x).cuda() for x in (a_bm, a_sg, a_ms))
    inv_ms = timed_device(3, i_bm, i_sg, i_ms)
    inv_info = bls.LastBatchInfo()
    got_bad = np.flatnonzero(d_res.cpu().numpy() != 1)
    assert np.array_equal(got_bad, bad_idx), "1 %-invalid leg: rejected rounds differ from the injected ones"
    nsig_valid = float(np.unpackbits(a_bm, axis=1, bitorder="little")[:, :N_COMMITTEE].sum()) - float(np.unpackbits(a_bm[bad_idx], axis=1, bitorder="little")[:, :N_COMMITTEE].sum())
    del i_bm, i_sg, i_ms

    # e2e: host buffers through the public C-ABI call, copies inside the timed region
    step_host(); torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    barrier()
    e2e_s = time.perf_counter() - t0
    assert int(h_res.sum().item()) == B
    clocks = sampler.finish()

    # batch-size sweep (BASELINE.md C2: B in {1, 64, 1 024, 16 384} rounds in flight) through the host-buffer call: latency and sigs/s
    sweep = {}
    spr = nsig / B
    bls.SetParam("hm_cache", 0)          # cold: every call hashes its message(s); the H(m) cache is measured separately below
    for bsz in (1, 64, 1024, 16384):
        if bsz > B: continue
        lat = []
        for _ in range(5 if bsz <= 1024 else 3):
            t0 = time.perf_counter()
            rc = L.hbls_aggregate_verify_batch(com.h, bsz, h_bm.data_ptr(), blen, h_sig.data_ptr(), h_msg.data_ptr(), MSG_LEN, h_res.data_ptr())
            lat.append((time.perf_counter() - t0) * 1e3)
        assert rc == 0 and int(h_res[:bsz].sum().item()) == bsz
        ms_ = float(np.median(lat))
        sweep[str(bsz)] = {"ms": ms_, "sigs_per_s": bsz * spr / (ms_ * 1e-3), "mode": bls.LastBatchInfo()["mode"]}
    single_round_ms = sweep["1"]["ms"]
    # informational: the leader's commit-phase vote collection (R9, consensus/leader.go:227-290): 250 individual
    # signatures on ONE payload, one device call (single-bit bitmaps; H(m) computed once)
    vmsg = msgs[:MSG_LEN]
    vsigs, vok = bls.SignHashBatch(b"".join(wl.sk_bytes(k) for k in sks), vmsg * N_COMMITTEE, MSG_LEN)
    vbm = bytearray(N_COMMITTEE * blen)
    for i in range(N_COMMITTEE): vbm[i * blen + (i >> 3)] |= 1 << (i & 7)
    vlat = []
    for _ in range(5):
        t0 = time.perf_counter()
        vres = com.AggregateVerifyBatch(bytes(vbm), vsigs, vmsg * N_COMMITTEE, MSG_LEN)
        vlat.append((time.perf_counter() - t0) * 1e3)
    assert vres == b"\x01" * N_COMMITTEE
    votes250_ms = float(np.median(vlat))
    # the same two calls with H(m) already in the library's device cache -- the node has SIGNED the message itself before it verifies
    # the aggregate over it (consensus/validator.go: prepare / commit vote, then :219-236), or prefetched it on ANNOUNCE
    bls.SetParam("hm_cache", 1)
    warm = {}
    for name, fn in (("single_round", lambda: L.hbls_aggregate_verify_batch(com.h, 1, h_bm.data_ptr(), blen, h_sig.data_ptr(), h_msg.data_ptr(), MSG_LEN, h_res.data_ptr())),
                     ("leader_250_votes", lambda: com.AggregateVerifyBatch(bytes(vbm), vsigs, vmsg * N_COMMITTEE, MSG_LEN))):
        bls.HashPrefetch(bytes(msgs[:MSG_LEN])); fn()
        wl_ = []
        for _ in range(5):
            t0 = time.perf_counter(); fn(); wl_.append((time.perf_counter() - t0) * 1e3)
        warm[name + "_hm_cached_ms"] = float(np.median(wl_))
    assert int(h_res[:1].sum().item()) == 1
    # SignHash of one key on one message (consensus/construct.go:101,110: the validator's prepare / commit vote): H(m) + the 255-bit ladder
    sk1 = bls.SecretKey(); sk1.Deserialize(wl.sk_bytes(sks[0]))
    def sign_ms(msg_of):
        ts = []
        for r in range(5):
            m_ = msg_of(r); t0 = time.perf_counter(); sg = sk1.SignHash(m_); ts.append((time.perf_counter() - t0) * 1e3)
            assert sg is not None
        return float(np.median(ts))
    warm["sign_hash_ms"] = sign_ms(lambda r: wl.commit_payload("bench/sign", r))                 # fresh message every call
    warm["sign_hash_hm_cached_ms"] = sign_ms(lambda r: bytes(msgs[:MSG_LEN]))
    warm["hash_cache"] = bls.HashCacheStats()

    others = None
    if not args.no_other_configs:
        others = other_configs(bls, world, rank, dist, "cuda")
    from harmony_b200 import shard
    dev_ms_max, e2e_ms_max, nsig_total = shard.reduce_step_stats(dev_ms, e2e_s * 1e3, float(nsig), device="cuda")
    if rank != 0:
        if world > 1: dist.destroy_process_group()
        return

    value = nsig_total * args.steps / (dev_ms_max * 1e-3)
    e2e_value = nsig_total * args.steps / (e2e_ms_max * 1e-3)

    # ---- roofline of the dominant kernel: the integer multiplier.  HBM is idle by construction (DESIGN.md).
    # Denominator (calibrated in round 2, profiles/r2_probe_int.*): a 32x32+64 MAC is one IMAD.WIDE, and an IMAD.WIDE holds the
    # FMA-heavy pipe of a scheduler for 4 cycles per warp (ncu: 4.0 pipe-cycles per instruction, carry-chained or not), so the chip
    # peak is SMs x 4 schedulers x 8 MAC/clk x SM clock.  The live probe (the multiplier's own carry chains, nothing else) reaches ~90 % of it.
    probe_macs, max_clock_hz = bls.ProbeMac32PerS(8192)
    sm_count = torch.cuda.get_device_properties(local).multi_processor_count
    sm_clock_hz = min(max_clock_hz, clocks["sm_mhz"] * 1e6) if clocks.get("sm_mhz") else max_clock_hz     # median SM clock sampled during the timed region
    peak = sm_count * 4 * 8 * sm_clock_hz
    binfo = bls.BuildInfo()
    names = list(bls.STAGE_NAMES)
    if B >= sm_count * 256: names[0] = "k_mask_aggregate_serial"
    rlc = bls.GetBatchMode() == 1 and B >= bls.GetParam("rlc_min")
    G = rlc_group_size(B, sm_count)
    if rlc:
        # batched form: slot 4 = coefficient scaling + group sums, slot 5 = (G+1)-pair Miller loop + ONE final exponentiation per group
        names[5] = f"k_rlc_pairing_split<{G}>"
        macs = executed_mac32_per_round(binfo["batch_inv"], G)
    else:
        t = EXEC_FP_OPS[bool(binfo["batch_inv"])]
        names[4], names[5] = "(unused)", "k_pairing_verify_split"
        macs = [mac32(t["mask"]), mac32((99, 381)), mac32(t["decode"]), mac32(t["hash"]), 0.0, mac32(EXACT_PAIRING_FP_OPS)]
    dom = int(np.argmax(stage_ms))
    dom_name, dom_macs, dom_ms = names[dom], macs[dom], stage_ms[dom]
    two_kernels = None
    if rlc and dom == 5 and lines_ms > 0:
        # the batched pairing stage ran as two kernels (running points + lines | accumulator + final exponentiation): the roofline is
        # that of the larger one, with its own executed work and its own CUDA-event time
        lm = mac32(EXEC_FP_OPS_LINES[G]) / G; am = macs[5] - lm; a_ms = stage_ms[5] - lines_ms
        two_kernels = {f"k_rlc_lines_split<{G}>": {"ms": lines_ms, "mac32_per_round": lm, "frac_of_peak": None},
                       f"k_rlc_accum_split<{G}>": {"ms": a_ms, "mac32_per_round": am, "frac_of_peak": None}}
        names[5] = f"k_rlc_lines_split<{G}>+k_rlc_accum_split<{G}>"
        dom_name, dom_macs, dom_ms = (f"k_rlc_accum_split<{G}>", am, a_ms) if a_ms >= lines_ms else (f"k_rlc_lines_split<{G}>", lm, lines_ms)
    achieved = dom_macs * B / (dom_ms * 1e-3)
    total_macs = sum(macs)
    step_s = dev_ms / args.steps * 1e-3
    bytes_per_round = blen + 96 + MSG_LEN + 1
    traffic = ncu_dram_bytes(dom_name.split("<")[0])
    orc = oracle_lib()
    S = min(B, 64)
    exact_macs = stage_mac32_per_round(orc, pks, bitmaps, sigs, msgs, blen, sample=min(12, S))     # the reference algorithm, oracle counter
    if two_kernels:
        for kk in two_kernels.values(): kk["frac_of_peak"] = kk["mac32_per_round"] * B / (kk["ms"] * 1e-3) / peak
    roofline = {"bound": "int32-imad", "kernel": dom_name, "achieved": achieved / 1e12, "peak": peak / 1e12, "unit": "TMAC32/s",
                "frac": achieved / peak,
                "peak_source": f"FMA-heavy pipe: {sm_count} SMs x 4 schedulers x 8 IMAD.WIDE MAC/clk x {sm_clock_hz / 1e9:.3f} GHz (median SM clock nvidia-smi reported during the timed region); "
                               "4 pipe-cycles per IMAD.WIDE warp instruction measured with ncu (profiles/r2_probe_int_ncu.txt)",
                "probe_achieved": probe_macs / 1e12, "probe_frac_of_peak": probe_macs / peak,
                "probe": "hbls_probe_mac32_per_s: the field multiplier's own mad.lo.cc/madc.hi.cc rows (IMAD.WIDE.U32.X), 4 independent accumulator sets per thread, 512 threads/SM",
                # DRAM bytes of ONE launch of the dominant kernel from the newest committed ncu --set full capture of this workload:
                # per-thread Fp12 temporaries spilling past L2, not input traffic
                "traffic": traffic[0] if traffic else None, "traffic_source": (traffic[1] + " (dram__bytes_read.sum + dram__bytes_write.sum)") if traffic else None,
                "algorithm": (f"random-linear-combination batch check, groups of {G} rounds (exact pass over the rounds of failed groups only)"
                              if rlc else "exact per-round FastAggregateVerify"),
                "work_counted": "EXECUTED Fp multiplications/squarings of the device code, all six stages (x300 / x234 MAC32 each; adds, shifts, selects not counted), "
                                "from the same kernels run on the host: tests/emu emu_stage_counts / emu_rlc_stage_counts",
                "kernel_mac32_per_round": dom_macs, "kernel_ms": dom_ms, "pairing_stage_kernels": two_kernels, "executed_mac32_per_round": total_macs,
                "pipeline_frac": total_macs * B / step_s / peak,
                "reference_algorithm_mac32_per_round": sum(exact_macs),
                "algorithmic_saving_vs_reference": 1.0 - total_macs / sum(exact_macs),
                "stage_ms_note": "per-kernel CUDA-event times from 3 extra passes after the timed region",
                "stage_ms": {n: float(m) for n, m in zip(names, stage_ms)},
                "stage_mac32_per_round": {n: m for n, m in zip(names, macs)},
                "stage_frac_of_peak": {n: (m * B / (t_ * 1e-3) / peak if t_ > 0.05 else None) for n, m, t_ in zip(names, macs, stage_ms)},
                "build": binfo,
                "hbm_algorithmic_gbs": bytes_per_round * B / step_s / 1e9}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        roofline["hbm_peak_gbs_measured"] = peaks.get("hbm_gbs")
    except Exception:
        roofline["hbm_peak_gbs_measured"] = None

    threads, core_info = usable_cores()
    cpu = None
    if world == 1:
        rps, done, good = cpu_rounds_per_s(orc, pks, bitmaps[:S * blen], sigs[:S * 96], msgs[:S * MSG_LEN], blen, 12.0, threads)
        rps1, done1, good1 = cpu_rounds_per_s(orc, pks, bitmaps[:S * blen], sigs[:S * 96], msgs[:S * MSG_LEN], blen, 4.0, 1)
        cpu = {"value": rps * spr, "unit": "sigs/s", "cores": threads, "kind": "port", "core_info": core_info,
               "sample": f"first {S} rounds of the same workload cycled for 12 s on {threads} threads ({done} rounds); restated CPU path oracle/hbls_oracle.c",
               "single_thread_value": rps1 * spr, "thread_scaling": rps / rps1 if rps1 else None, "all_correct": bool(good and good1),
               "reference_published_ms": {"VerifyHash": 1.5, "Sign.Deserialize": 0.52, "src": "reference test/chain/vrf/main.go:109-112, test/chain/reward/main.go:239-245 (hardware unspecified)"}}

    line = {"metric": "BLS aggregate-verify sigs/sec (250-validator FBFT commit batch)", "value": value, "unit": "sigs/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (12x32-bit Montgomery limbs, IMAD.WIDE)",
            "data": "synthetic",
            "config": {"workload": "FBFT commit-phase: 250-validator committee, single message per round, FastAggregateVerify per round (BASELINE configs[1]), " + f"{world}xB200",
                       "committee": N_COMMITTEE, "rounds_per_step_per_gpu": B, "signers_per_round": "167/200/250 cycling", "msg_len": MSG_LEN,
                       "sharding": "rounds by index, no data-path collective", "l2": "256 MiB flush between timed steps",
                       "timing": "CUDA events per step on the launching stream, max over ranks"},
            "e2e": {"value": e2e_value, "unit": "sigs/s", "h2d_bytes_per_step": B * (blen + 96 + MSG_LEN), "d2h_bytes_per_step": B,
                    "ms_per_step": e2e_ms_max / args.steps, "api": "hbls_aggregate_verify_batch (pinned host buffers)"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "wall_s_timed_region": t_wall,
            "value_1pct_invalid": nsig_valid / (inv_ms * 1e-3),
            "one_pct_invalid": {"ms_per_step": inv_ms, "invalid_rounds": int(n_bad), "kinds": "wrong payload / other round's signature / flipped bitmap bit / undecodable signature",
                                "value_this_rank": nsig_valid / (inv_ms * 1e-3), "unit": "sigs/s (constituent signatures of the rounds that verify)",
                                "results_exact": True, "batch_info": inv_info},
            "exact_mode": {"ms_per_step": exact_ms, "value_this_rank": nsig / (exact_ms * 1e-3), "unit": "sigs/s",
                           "note": "hbls_set_batch_mode(0): every round verified on its own (no random linear combination), rank 0, 3 steps"},
            "batch_sweep_e2e": sweep,
            "single_round_latency_ms": single_round_ms, "leader_250_votes_same_msg_latency_ms": votes250_ms, "latency_hm_cached": warm}
    if cpu: line["cpu_baseline"] = cpu
    if others: line["other_configs"] = others
    print(json.dumps(line), flush=True)
    if world > 1: dist.destroy_process_group()

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=303104, help="rounds per step per GPU (default: 37 888 groups of 8 = one lane pair per group on 148 SMs x 512 threads)")
    ap.add_argument("--impl", default="hbls", choices=["hbls", "reference"])
    ap.add_argument("--no-other-configs", action="store_true", help="skip the short C3 / C4 / C5 legs (BASELINE configs[2..4]) reported beside the headline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the per-round results of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "hbls":
        ap.error("--dump-outputs needs --impl hbls")
    if args.warmup < 3 and args.impl == "hbls":
        log("note: warm-up < 3 steps requested")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)

if __name__ == "__main__":
    main()
