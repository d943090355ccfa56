"""Dispatch-path coverage of the batch verifier.

launch_verify_tail / agg_verify_device_locked (harmony_b200/csrc/hbls.cu) pick one of many kernel paths for the same answer, by
batch size, SM count and the hbls_set_param knobs.  Each test here runs one path (or both sides of one switch), checks the per-round
booleans against a vector known by construction and against the CPU oracle (every bad round, every round that shares a batched group
with one, a seeded sample), and proves that the two calls of a pair took different paths: the kernel-launch count, hbls_last_batch_info
or the set of kernels that ran differ.  Thresholds that scale with the chip are derived from the device's SM count the way hbls.cu
derives them; the two-phase chunk (RLC_CHUNK_GROUPS) is a constant.
"""
import json, os, random, re, tempfile
from types import SimpleNamespace
import pytest
from harmony_b200 import workload as wl

pytestmark = pytest.mark.gpu

P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
R = wl.R_ORDER
RLC_CHUNK_GROUPS = 37888           # hbls.cu: groups per pass of the two-phase pairing
HB_RLC_GMAX = 8                    # kernels.cuh: largest batched group; batches under 2 * HB_RLC_GMAX rounds are never grouped
HB_MASK_LIST = 512                 # kernels.cuh: k_mask_aggregate_serial sums from an index list when one side has <= 512 bits
# every name hbls_set_param accepts (include/hbls.h and param_slot in hbls.cu)
KNOBS = ("rlc_min", "rlc_g", "tpsm", "tpsm_split", "tpsm_light", "coop_max", "overlap", "coop_wpsm", "hm_cache", "hash_coop_max",
         "mask_sort", "hash_split", "hash_fallback", "rlc_two_phase", "tpsm_cof", "tpsm_dec", "tpsm_scale", "tpsm_scale_g1",
         "scale_split", "decode_split", "exact_two_phase", "tpsm_lines", "tpsm_accum", "tpsm_sw")
KINDS = ("wrong_msg", "swapped_sig", "flipped_bitmap_bit", "undecodable_sig", "identity_sig", "empty_bitmap")
POOL = 8 * (RLC_CHUNK_GROUPS + 512) + 5      # 307 205 signed rounds: every batch below is a prefix of this pool


# ------------------------------------------------------------------------------------------------------------------ infrastructure
@pytest.fixture(scope="module")
def defaults(gbls):
    """Batch mode and every knob as the library started with them (each name round-trips through hbls_set_param)."""
    params = {k: gbls.GetParam(k) for k in KNOBS}
    for k, v in params.items():
        gbls.SetParam(k, v)
    return gbls.GetBatchMode(), params

def reset_knobs(gbls, defaults):
    mode, params = defaults
    for k, v in params.items():
        gbls.SetParam(k, v)
    gbls.SetBatchMode(mode)

@pytest.fixture(autouse=True)
def restore_knobs(gbls, defaults):
    """Put the snapshot back after every test, also after a failure."""
    yield
    reset_knobs(gbls, defaults)

@pytest.fixture(scope="module")
def sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count

def set_knobs(gbls, **kv):
    for k, v in kv.items():
        if k == "mode": gbls.SetBatchMode(v)
        else: gbls.SetParam(k, v)

def call(gbls, fn):
    """(result, kernels launched, hbls_last_batch_info, H(m) cache lookups) of one library call."""
    c0 = gbls.KernelLaunchCount(); h0 = gbls.HashCacheStats()
    out = fn()
    h1 = gbls.HashCacheStats()
    return SimpleNamespace(res=out, launches=gbls.KernelLaunchCount() - c0, info=gbls.LastBatchInfo(),
                           lookups=h1["hits"] + h1["misses"] - h0["hits"] - h0["misses"])

def path_of(r):
    """What identifies a path: launches, form (mode, G, CTA size) and H(m) cache lookups -- not the size-dependent counters."""
    i = r.info
    return (r.launches, i["mode"], i["group_size"], i["cta_threads"], r.lookups)

def assert_other_path(a, b, what):
    assert path_of(a) != path_of(b), f"{what}: both calls took the same path ({a.launches} launches, {a.info})"

def kernels_run(fn):
    """Names of the kernels a call launched (CUPTI through torch.profiler), for switches that change a kernel but not the launch count."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)
    names = {e.get("name", "") for e in (ev["traceEvents"] if isinstance(ev, dict) else ev) if e.get("cat") == "kernel"}
    return out, names

def ran(names, kernel):
    return any(re.search(r"(^|[\s:])" + re.escape(kernel) + r"[(<]", n) for n in names)


class Oracle:
    """CPU oracle verdicts, memoised: the batches below share their rounds with each other."""
    def __init__(self, oracle):
        self.o = oracle; self.memo = {}
    def verdict(self, och, bm, sg, mm):
        key = (och, bytes(bm), bytes(sg), bytes(mm))
        if key not in self.memo:
            self.memo[key] = self.o.committee_aggregate_verify(och, key[1], key[2], key[3]) == 1
        return self.memo[key]

@pytest.fixture(scope="module")
def orc(oracle):
    return Oracle(oracle)

def make_committee(gbls, oracle, sks, pks=None):
    if pks is None:
        blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
        pks = [blob[48 * i:48 * i + 48] for i in range(len(sks))]
    n = len(pks)
    return SimpleNamespace(sks=sks, pks=pks, com=gbls.Committee(pks), och=oracle.committee(pks), n=n, blen=(n + 7) >> 3)

@pytest.fixture(scope="module")
def bench_com(gbls, oracle):
    import bench
    return make_committee(gbls, oracle, bench.make_committee_sks())

@pytest.fixture(scope="module")
def pool(gbls, bench_com):
    """POOL rounds of the benchmark committee: 16 distinct bitmaps (167 / 200 / 250 signers) cycled, distinct random payloads."""
    import numpy as np
    c = bench_com
    bms = [wl.bitmap_with_k("paths", j, c.n, (167, 200, 250)[j % 3]) for j in range(16)]
    agg = [wl.sk_bytes(wl.round_signer_sum(c.sks, bm)) for bm in bms]
    reps = POOL // 16 + 1
    msgs = np.random.default_rng(2026).integers(0, 256, POOL * 48, dtype=np.uint8).tobytes()
    sigs, ok = gbls.SignHashBatch((b"".join(agg) * reps)[:32 * POOL], msgs, 48)
    assert ok == b"\x01" * POOL
    return SimpleNamespace(c=c, bms=bms, agg=agg, bitmaps=(b"".join(bms) * reps)[:c.blen * POOL], sigs=sigs, msgs=msgs)


class Batch:
    """The first B rounds of a signed pool, with bad rounds planted at known positions."""
    def __init__(self, pool, B, msg_len=48):
        self.pool, self.c, self.B, self.L = pool, pool.c, B, msg_len
        self.bm = bytearray(pool.bitmaps[:pool.c.blen * B]); self.sg = bytearray(pool.sigs[:96 * B])
        self.mm = bytearray(pool.msgs[:msg_len * B]); self.bad = {}
    def corrupt(self, j, kind):
        bl, L = self.c.blen, self.L
        if kind == "wrong_msg": self.mm[L * j + min(17, L - 1)] ^= 0x20
        elif kind == "swapped_sig":
            o = (j + 1) % (len(self.pool.sigs) // 96); self.sg[96 * j:96 * j + 96] = self.pool.sigs[96 * o:96 * o + 96]
        elif kind == "flipped_bitmap_bit": self.bm[bl * j + j % (bl - 1)] ^= 0x04
        elif kind == "undecodable_sig": self.sg[96 * j:96 * j + 96] = b"\xff" * 96
        elif kind == "identity_sig": self.sg[96 * j:96 * j + 96] = bytes(96)
        elif kind == "empty_bitmap": self.bm[bl * j:bl * j + bl] = bytes(bl)
        else: raise AssertionError(kind)
        self.bad[j] = kind
    def plant(self, positions, kinds=KINDS):
        for t, j in enumerate(sorted(set(positions))):
            self.corrupt(j, kinds[t % len(kinds)])
        return self
    def expected(self):
        e = bytearray(b"\x01" * self.B)
        for j in self.bad: e[j] = 0
        return bytes(e)
    def round(self, j):
        bl, L = self.c.blen, self.L
        return self.bm[bl * j:bl * j + bl], self.sg[96 * j:96 * j + 96], self.mm[L * j:L * j + L]
    def verify(self, gbls):
        return call(gbls, lambda: self.c.com.AggregateVerifyBatch(bytes(self.bm), bytes(self.sg), bytes(self.mm), self.L))

def spread(B, extra=()):
    """Bad-round positions at both ends, the middle and the thirds of a batch."""
    return sorted({j for j in (0, B // 3, B // 2, 2 * B // 3, B - 2, B - 1, *extra) if 0 <= j < B})

def check(orc, batch, r, sample=24, seed=0, mate_groups=None):
    """Booleans == the vector known by construction; the oracle agrees on every bad round, every round that shares a batched group
    with one (the first `mate_groups` bad groups when given) and a seeded sample."""
    exp = batch.expected()
    if r.res != exp:
        diff = [j for j in range(batch.B) if r.res[j] != exp[j]]
        raise AssertionError(f"{len(diff)} wrong verdicts, first {diff[:10]} (planted: {[(j, batch.bad.get(j)) for j in diff[:10]]}), info {r.info}")
    idx = set(batch.bad)
    info = r.info
    if info["mode"] == 1 and info["groups"]:
        G, ng = info["group_size"], info["groups"]
        groups = sorted({j % ng for j in batch.bad if j < G * ng})
        for g in groups[:mate_groups]:
            idx |= {g + k * ng for k in range(G)}
    idx |= set(random.Random(seed).sample(range(batch.B), min(sample, batch.B)))
    for j in sorted(idx):
        assert (r.res[j] == 1) == orc.verdict(batch.c.och, *batch.round(j)), (j, batch.bad.get(j), r.res[j])


# ------------------------------------------------------------------------------------------------------- A. chunk boundaries
def group_round(ng, g, k):
    return k * ng + g          # strided groups: round of (position k, group g)

@pytest.mark.parametrize("G, extra_groups, tail", [(4, 300, 3), (8, 512, 5)])
def test_two_chunk_batched_pairing(gbls, orc, pool, sm, G, extra_groups, tail):
    """G = 4 at B = 4 (37 888 + 300) + 3 and G = 8 at B = 8 (37 888 + 512) + 5 (default knobs): the two-phase pairing runs a second
    chunk with the group offset g0 > 0.  Bad rounds sit in group 0, the last group of the first chunk, the first group of the second
    chunk, the last group, and the tail.  groups_failed pins that the batched test itself (not only the exact pass) got every group
    right: a second chunk reading the first chunk's points would fail its groups and still return the right booleans."""
    ng = RLC_CHUNK_GROUPS + extra_groups
    B = G * ng + tail
    assert (2 * (B // 8) >= sm * 512) == (G == 8), "the default G for this B is derived from the SM count"
    b = Batch(pool, B)
    bad_groups = [0, RLC_CHUNK_GROUPS - 1, RLC_CHUNK_GROUPS, ng - 1]
    b.plant([group_round(ng, g, (i + 1) % G) for i, g in enumerate(bad_groups)] + [G * ng + tail - 1])
    r = b.verify(gbls)
    assert r.info["mode"] == 1 and r.info["group_size"] == G and r.info["groups"] == ng and r.info["tail_rounds"] == tail
    assert r.info["groups_failed"] == len(bad_groups) and r.info["rounds_rechecked"] == G * len(bad_groups)
    check(orc, b, r)

def test_exact_list_pass_over_two_chunks(gbls, orc, pool):
    """B = 303 104 (G = 8) with 4 800 bad rounds in distinct groups: 38 400 listed rounds, so the exact pass over failed groups
    (k_rlc_lines_split<1> / k_rlc_accum_split<1> over the device-side list) runs two chunks.  Exactly the bad rounds are 0; then the
    same batch through the one-kernel list pass (exact_two_phase 0) gives the same bytes."""
    B, G = 8 * RLC_CHUNK_GROUPS, 8
    ng = B // G
    rng = random.Random(48)
    groups = rng.sample(range(ng), 4800)
    b = Batch(pool, B)
    for g in groups:
        b.corrupt(group_round(ng, g, rng.randrange(G)), "wrong_msg")
    r = b.verify(gbls)
    assert r.info["group_size"] == G and r.info["groups_failed"] == len(groups)
    assert r.info["rounds_rechecked"] == G * len(groups) > RLC_CHUNK_GROUPS
    check(orc, b, r, mate_groups=24)
    set_knobs(gbls, exact_two_phase=0)
    r0 = b.verify(gbls)
    assert r0.res == r.res
    assert_other_path(r, r0, "exact_two_phase 1 | 0 in the failed-groups pass")

def test_mode0_exact_two_phase_two_chunks(gbls, orc, pool):
    """Mode 0 beyond coop_max at B = 37 888 + 517: the exact check runs as k_rlc_lines_split<1> / k_rlc_accum_split<1> in two chunks.
    Bad rounds at 37 887, 37 888 and B - 1; the one-kernel form (exact_two_phase 0) must agree."""
    B = RLC_CHUNK_GROUPS + 517
    b = Batch(pool, B).plant([RLC_CHUNK_GROUPS - 1, RLC_CHUNK_GROUPS, B - 1, 5, 20000])
    set_knobs(gbls, mode=0)
    r = b.verify(gbls)
    assert r.info["mode"] == 0
    check(orc, b, r)
    set_knobs(gbls, exact_two_phase=0)
    r0 = b.verify(gbls)
    assert r0.res == r.res
    assert_other_path(r, r0, "mode 0: exact_two_phase 1 | 0")


# ------------------------------------------------------------------------------------------------------- B. size thresholds
def threshold_cases(sm):
    S256 = 256 * sm
    return [
        # (left B, right B, knobs, what switches)
        (1, 2, {}, None, "one round: H(m) of the single message through the cache | per-round hash"),
        (15, 16, {"rlc_min": 1}, None, "2 * HB_RLC_GMAX floor of the batched form (rlc_min lowered to reach it at 15 | 16)"),
        (592, 593, {}, ("k_hash_to_g2_coop", "k_hash_to_g2_pair"), "hash_coop_max: warp per message | lane pair per message"),
        (4096, 4097, {}, None, "coop_max: warp-per-round latency form | exact lane-pair form"),
        (12287, 12288, {}, None, "rlc_min: exact | batched groups"),
        # one tail of 3 rounds less on the right costs as many launches as the counting sort adds: named kernels prove the switch
        (S256 - 1, S256, {}, ("k_mask_aggregate", "k_mask_aggregate_serial"), "serial mask kernel from 256 * SM rounds"),
        (S256 - 1, S256, {"mode": 0}, None, "full-chip lock-stepped exact CTAs from 2B >= 512 * SM"),
        (4 * S256 - 1, 4 * S256, {}, None, "full-chip batched pairing from ng >= 256 * SM (G = 4)"),
        (8 * S256 - 1, 8 * S256, {}, None, "G = 4 | 8 at B / 8 >= 256 * SM"),
    ]

@pytest.mark.parametrize("case", range(9))
def test_size_threshold_both_sides(gbls, orc, pool, sm, case):
    """Both sides of every size switch of the dispatcher, each batch with bad rounds of every kind; the two calls of a pair must
    take different paths and both give the expected bytes."""
    left, right, knobs, named, what = threshold_cases(sm)[case]
    set_knobs(gbls, **knobs)
    runs = []
    for side, B in enumerate((left, right)):
        b = Batch(pool, B).plant(spread(B, extra=(B // 5, B // 7)))
        if named:
            r, names = kernels_run(lambda: b.verify(gbls))
            assert ran(names, named[side]) and not ran(names, named[1 - side]), (what, B, sorted(names))
        else:
            r = b.verify(gbls)
        check(orc, b, r, sample=16, seed=B)
        runs.append(r)
    if not named:
        assert_other_path(runs[0], runs[1], what)
    if left == 1:        # a lone valid round as well
        b = Batch(pool, 1)
        assert b.verify(gbls).res == b"\x01"

SAME_MSG_CASES = {"latency": 300, "exact": 5000, "batched": 13000}

@pytest.mark.parametrize("regime", list(SAME_MSG_CASES))
def test_same_message_form(gbls, orc, pool, regime):
    """One message for the whole batch: H(m) once + k_broadcast_hm, in the latency (cold and warm H(m) cache), exact (beyond
    coop_max) and batched regimes.  Compared with a distinct-message batch of the same size, which takes the per-round hash."""
    c = pool.c
    B = SAME_MSG_CASES[regime]
    msg = wl.commit_payload("same/" + regime, B)
    sigs16, ok = gbls.SignHashBatch(b"".join(pool.agg), msg * 16, 48)
    assert ok == b"\x01" * 16
    reps = B // 16 + 1
    same = SimpleNamespace(c=c, bms=pool.bms, agg=pool.agg, bitmaps=(b"".join(pool.bms) * reps)[:c.blen * B],
                           sigs=(sigs16 * reps)[:96 * B], msgs=msg * B)
    b = Batch(same, B).plant(spread(B, extra=(B // 5,)), kinds=KINDS[1:])     # every kind but a changed message
    if regime == "latency":
        h0 = gbls.HashCacheStats()
        cold = b.verify(gbls)
        h1 = gbls.HashCacheStats()
        warm = b.verify(gbls)
        h2 = gbls.HashCacheStats()
        assert h1["misses"] - h0["misses"] == 1 and h2["hits"] - h1["hits"] == 1
        assert cold.res == warm.res
        assert_other_path(cold, warm, "cold | warm H(m) cache")
        r = warm
    else:
        r = b.verify(gbls)
    assert r.info["mode"] == (1 if regime == "batched" else 0)
    check(orc, b, r, sample=16)
    d = Batch(pool, B).plant(spread(B))
    rd = d.verify(gbls)
    check(orc, d, rd, sample=8)
    assert_other_path(r, rd, f"{regime}: same message | distinct messages")


# ------------------------------------------------------------------------------------------------------------- C. knob matrix
# One mid-size batch per regime.  Lowered thresholds reach the regime at a size that keeps the oracle sample cheap:
#   exact   -- coop_max lowered to 1 024, B = 1 500 in mode 0 (beyond the warp-per-round form, below the batched form);
#   batched -- rlc_min lowered to 1 024, B = 2 053 (G = 4 and 8 both leave a tail of 1 or 5 rounds).
REGIMES = {
    "latency": (300, {}),
    "exact": (1500, {"coop_max": 1024}),
    "batched": (2053, {"rlc_min": 1024}),
}
SWEEP = {
    "latency": [("overlap", 0), ("hash_coop_max", 0), ("hash_fallback", 1)],
    "exact": [("hash_split", 0), ("hash_split", 1), ("decode_split", 0), ("exact_two_phase", 0), ("rlc_two_phase", 1), ("rlc_two_phase", 0)],
    "batched": [("hash_split", 0), ("hash_split", 1), ("scale_split", 0), ("decode_split", 0), ("exact_two_phase", 0),
                ("rlc_two_phase", 1), ("rlc_two_phase", 0), ("rlc_g", 8)],
}
# same launch count on both sides: the kernel that must (not) have run instead
NAMED = {("hash_coop_max", 0): ("k_hash_to_g2_coop", "k_hash_to_g2_pair")}

@pytest.mark.parametrize("regime", list(REGIMES))
def test_knob_sweep(gbls, orc, pool, regime):
    """Each knob moved away from its default, one at a time: identical bytes, equal to the expected vector, on another path.
    hash_fallback is a kernel argument (the warp-per-message hash takes its complete-formula branch), not another launch, so only
    its bytes are compared."""
    B, knobs = REGIMES[regime]
    set_knobs(gbls, **knobs)
    b = Batch(pool, B).plant(spread(B, extra=(B // 5, B // 9, B // 11)))
    base = b.verify(gbls)
    check(orc, b, base, sample=24)
    assert base.info["mode"] == (1 if regime == "batched" else 0)
    for name, value in SWEEP[regime]:
        old = gbls.GetParam(name)
        assert old != value, (name, value)
        set_knobs(gbls, **{name: value})
        try:
            if (name, value) in NAMED:
                r, names = kernels_run(lambda: b.verify(gbls))
                before, after = NAMED[(name, value)]
                assert ran(names, after) and not ran(names, before), (name, value, sorted(names))
            else:
                r = b.verify(gbls)
                if name != "hash_fallback":
                    assert_other_path(base, r, f"{regime}: {name} {old} | {value}")
        finally:
            set_knobs(gbls, **{name: old})
        assert r.res == base.res, (regime, name, value)

def test_batched_pairwise_combinations(gbls, orc, pool):
    """rlc_g x rlc_two_phase x exact_two_phase in the batched regime: k_rlc_pairing_split<4 / 8> (fused) and k_rlc_lines_split /
    k_rlc_accum_split<4 / 8>, each with the two-kernel or the one-kernel exact pass over failed groups; tails of 1 to 7 rounds."""
    set_knobs(gbls, rlc_min=1024)
    # below the full-chip size rlc_two_phase 0 and 1 both keep the fused kernel, and exact_two_phase only matters with the two-kernel
    # pairing: three paths per G, six in all, each reached by every combination of its class and by no other
    cls = lambda G, two, ex: (G, two >= 2, two >= 2 and ex == 1)
    for tail in (1, 3, 7):
        paths = {}
        B = 8 * 256 + tail
        b = Batch(pool, B).plant(spread(B, extra=(7, 300, 301, 8 * 256)))
        results = set()
        for G in (4, 8):
            for two in (0, 1, 2):
                for ex in (0, 1):
                    set_knobs(gbls, rlc_g=G, rlc_two_phase=two, exact_two_phase=ex)
                    r = b.verify(gbls)
                    assert r.info["group_size"] == G and r.info["tail_rounds"] == B % G
                    assert r.res == b.expected(), (tail, G, two, ex)
                    results.add(r.res)
                    paths.setdefault(cls(G, two, ex), set()).add(path_of(r))
        check(orc, b, r, sample=8, seed=tail)
        assert len(results) == 1
        assert len(paths) == 6 and all(len(v) == 1 for v in paths.values()), paths
        assert len({next(iter(v)) for v in paths.values()}) == 6, paths

def test_two_phase_at_full_chip(gbls, orc, pool, sm):
    """At ng >= 256 * SM groups (G = 4) rlc_two_phase 1 switches to the two-kernel pairing; 0 keeps the fused 512-thread kernel."""
    B = 4 * 256 * sm + 3
    b = Batch(pool, B).plant(spread(B, extra=(1, 2, 3)))
    runs = {}
    for two in (0, 1):
        set_knobs(gbls, rlc_two_phase=two)
        runs[two] = b.verify(gbls)
        assert runs[two].info["cta_threads"] == 512 and runs[two].info["group_size"] == 4
    assert runs[0].res == runs[1].res
    check(orc, b, runs[1], sample=16)
    assert_other_path(runs[0], runs[1], "full chip: rlc_two_phase 0 | 1")

def test_mask_sort_large_batch(gbls, orc, pool, sm):
    """mask_sort 0 | 1 at B = 256 * SM (serial mask kernel with and without the counting sort of rounds by addition count)."""
    B = 256 * sm
    b = Batch(pool, B).plant(spread(B, extra=(17, 18, 19, 20, 21, 22)))
    runs = {}
    for s in (1, 0):
        set_knobs(gbls, mask_sort=s)
        runs[s] = b.verify(gbls)
    assert runs[0].res == runs[1].res
    check(orc, b, runs[0], sample=16)
    assert_other_path(runs[0], runs[1], "mask_sort 0 | 1")

@pytest.fixture(scope="module")
def triples(gbls):
    k = 5000
    sks = b"".join(wl.sk_bytes(wl.seeded_sk("paths/t", i)) for i in range(k))
    msgs = b"".join(wl.seeded_bytes("paths/t/m", i, 32) for i in range(k))
    pks = gbls.GetPublicKeyBatch(sks)
    sigs, ok = gbls.SignHashBatch(sks, msgs, 32)
    assert ok == b"\x01" * k
    return SimpleNamespace(k=k, pks=pks, sigs=sigs, msgs=msgs)

def test_verify_batch_batched_scale_split(gbls, oracle, triples):
    """VerifyBatch in the batched regime with undecodable and swapped keys: ok_pk enters k_rlc_scale but not k_rlc_scale_g1, so
    scale_split 0 and 1 must agree, with each other, with the exact mode and with the oracle."""
    k = 2053
    pk = bytearray(triples.pks[:48 * k]); sg = bytearray(triples.sigs[:96 * k]); mm = bytearray(triples.msgs[:32 * k])
    bad = {}
    for t, i in enumerate(spread(k, extra=(1, 2, 513, 514, 1026, 1027, 1540))):
        kind = ("pk_undecodable", "pk_swapped", "sig_undecodable", "wrong_msg", "pk_identity")[t % 5]
        bad[i] = kind
        if kind == "pk_undecodable": pk[48 * i:48 * i + 48] = b"\xff" * 48
        elif kind == "pk_swapped": o = (i + 3) % k; pk[48 * i:48 * i + 48] = triples.pks[48 * o:48 * o + 48]
        elif kind == "sig_undecodable": sg[96 * i:96 * i + 96] = b"\xff" * 96
        elif kind == "wrong_msg": mm[32 * i + 4] ^= 1
        else: pk[48 * i:48 * i + 48] = bytes(48)
    exp = bytes(0 if i in bad else 1 for i in range(k))
    set_knobs(gbls, rlc_min=1024)
    runs = {}
    for s in (1, 0):
        set_knobs(gbls, scale_split=s)
        runs[s] = call(gbls, lambda: gbls.VerifyBatch(bytes(pk), bytes(sg), bytes(mm), 32))
        assert runs[s].info["mode"] == 1
        assert runs[s].res == exp, (s, [i for i in range(k) if runs[s].res[i] != exp[i]][:10])
    assert_other_path(runs[0], runs[1], "VerifyBatch: scale_split 0 | 1")
    set_knobs(gbls, mode=0)
    assert gbls.VerifyBatch(bytes(pk), bytes(sg), bytes(mm), 32) == exp
    for i in sorted(set(bad) | set(random.Random(3).sample(range(k), 24))):
        assert oracle.verify_hash(bytes(sg[96 * i:96 * i + 96]), bytes(pk[48 * i:48 * i + 48]), bytes(mm[32 * i:32 * i + 32])) == (exp[i] == 1), i

def test_rlc_partial_above_coop_max(gbls, triples):
    """RlcPartial / RlcFold at k = 5 000 (above coop_max: k_g2_decode + k_hash_to_g2 + per-item k_rlc_scale): a valid slice folds to
    True, one bad item anywhere (wrong message, swapped signature) to False."""
    k = triples.k
    assert k > gbls.GetParam("coop_max")
    rec = gbls.RlcPartial(triples.pks, triples.sigs, triples.msgs, 32)
    assert gbls.RlcFold([rec]) is True
    mm = bytearray(triples.msgs); mm[32 * (k - 1) + 7] ^= 1
    assert gbls.RlcFold([gbls.RlcPartial(triples.pks, triples.sigs, bytes(mm), 32)]) is False
    sg = bytearray(triples.sigs); sg[96 * 2500:96 * 2501] = triples.sigs[96 * 2501:96 * 2502]
    assert gbls.RlcFold([gbls.RlcPartial(triples.pks, bytes(sg), triples.msgs, 32)]) is False


# ------------------------------------------------------------------------------------------------- D. degenerate group-law inputs
def bitmap_of(n, idx, pad=False):
    bm = bytearray((n + 7) >> 3)
    for i in idx: bm[i >> 3] |= 1 << (i & 7)
    if pad and n % 8: bm[-1] |= (0xff << (n % 8)) & 0xff
    return bytes(bm)

DEGEN_N = 300
IDENTITY_ROW = 299

@pytest.fixture(scope="module")
def degen(gbls, oracle):
    """300 keys with equal and opposite rows placed where one addition of each aggregation kernel meets them:
    rows 8 / 40 equal (one lane of the warp kernel, lane distance 32), 72 / 200 equal (one thread of k_g1_sum, distance 128),
    0 / 16 equal and 1 / 17 opposite (partners in the first level of the warp shuffle tree), 5 / 69 opposite (one lane),
    104 = -row 8 (P + P - P in lane 8), and an identity row."""
    n = DEGEN_N
    sks = [wl.seeded_sk("paths/degen", i) for i in range(n)]
    sks[40] = sks[8]; sks[200] = sks[72]; sks[16] = sks[0]
    sks[17] = (R - sks[1]) % R; sks[69] = (R - sks[5]) % R; sks[104] = (R - sks[8]) % R
    sks[IDENTITY_ROW] = 0
    blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
    pks = [blob[48 * i:48 * i + 48] for i in range(n)]
    pks[IDENTITY_ROW] = bytes(48)                  # the identity encoding; the oracle's committee accepts it
    assert oracle.pk_check(bytes(48))
    c = make_committee(gbls, oracle, sks, pks)
    every = set(range(n)); rnd = random.Random(9)
    some = set(rnd.sample(range(n), 100))
    sets = {
        "2P lane": {8, 40}, "P-P lane": {5, 69}, "P+P-P lane": {8, 40, 104}, "2P tree": {0, 16}, "P-P tree": {1, 17},
        "2P thread": {72, 200}, "identity row": {IDENTITY_ROW}, "identity row + key": {IDENTITY_ROW, 3}, "all": every,
        "all but 2P": every - {8, 40}, "all but P-P": every - {5, 69}, "all but P+P-P": every - {8, 40, 104},
        "all but 2P thread": every - {72, 200}, "empty": set(), "mixed": some | {0, 16, 1, 17, 5, 69, 8, 40, 104, 72, 200, IDENTITY_ROW},
        "mixed but P-P": (some | {5, 69}) - {1, 17, 8, 40},
    }
    names = list(sets)
    bms = [bitmap_of(n, sets[k], pad=(t % 2 == 1)) for t, k in enumerate(names)]
    sums = [sum(sks[i] for i in sets[k]) % R for k in names]
    msgs = [wl.commit_payload("paths/degen", t) for t in range(len(names))]
    sigs, ok = gbls.SignHashBatch(b"".join(wl.sk_bytes(s) for s in sums), b"".join(msgs), 48)
    sigs = [sigs[96 * t:96 * t + 96] if sums[t] else bytes(96) for t in range(len(names))]   # identity key: the identity signature
    return SimpleNamespace(c=c, names=names, sets=sets, bms=bms, sums=sums, msgs=msgs, sigs=sigs)

def test_degenerate_committee_mask_aggregate(gbls, oracle, degen):
    """Single-round MaskAggregate and the committee total (k_g1_sum) through equal / opposite rows; the identity key rules."""
    c = degen.c
    for name, bm in zip(degen.names, degen.bms):
        assert c.com.MaskAggregate(bm) == oracle.committee_mask_aggregate(c.och, bm), name
    assert c.com.MaskAggregate(degen.bms[degen.names.index("P-P lane")]) == bytes(48)
    assert c.com.MaskAggregate(degen.bms[degen.names.index("2P lane")]) == oracle.pk_add(c.pks[8], c.pks[8])

def degen_expected(degen):
    return bytes(1 if s else 0 for s in degen.sums)

def test_degenerate_committee_verdicts_small(gbls, orc, degen):
    """Warp kernel (small B), AggregateVerifyItems and the single-round entry: a round whose key sum is the identity is 0 on every path."""
    c = degen.c
    exp = degen_expected(degen)
    assert exp.count(0) >= 4
    ora = bytes(1 if orc.verdict(c.och, bm, s, m) else 0 for bm, s, m in zip(degen.bms, degen.sigs, degen.msgs))
    assert ora == exp
    res = c.com.AggregateVerifyBatch(b"".join(degen.bms), b"".join(degen.sigs), b"".join(degen.msgs), 48)
    assert res == exp
    res = gbls.AggregateVerifyItems([c.com] * len(degen.bms), degen.bms, b"".join(degen.sigs), b"".join(degen.msgs), 48)
    assert res == exp
    for bm, s, m, e in zip(degen.bms, degen.sigs, degen.msgs, exp):
        assert c.com.AggregateVerify(bm, s, m) == (e == 1)

@pytest.mark.parametrize("mask_sort", [1, 0])
def test_degenerate_committee_serial_kernel(gbls, orc, degen, sm, mask_sort):
    """B = 256 * SM rounds cycling over the degenerate bitmaps: k_mask_aggregate_serial (index list and complement sum over the
    committee total), with and without the counting sort."""
    import numpy as np
    c = degen.c
    B = 256 * sm
    nb = len(degen.bms)
    msgs = np.random.default_rng(77).integers(0, 256, B * 48, dtype=np.uint8).tobytes()
    sks = b"".join(wl.sk_bytes(degen.sums[j % nb]) for j in range(B))
    sigs, ok = gbls.SignHashBatch(sks, msgs, 48)
    sg = bytearray(sigs)
    for j in range(B):
        if not degen.sums[j % nb]: sg[96 * j:96 * j + 96] = bytes(96)
    bitmaps = (b"".join(degen.bms) * (B // nb + 1))[:c.blen * B]
    exp = (degen_expected(degen) * (B // nb + 1))[:B]
    set_knobs(gbls, mask_sort=mask_sort)
    r = call(gbls, lambda: c.com.AggregateVerifyBatch(bitmaps, bytes(sg), msgs, 48))
    assert r.res == exp, [j for j in range(B) if r.res[j] != exp[j]][:10]
    for j in list(range(nb)) + random.Random(4).sample(range(B), 16):
        assert (r.res[j] == 1) == orc.verdict(c.och, bitmaps[c.blen * j:c.blen * (j + 1)], sg[96 * j:96 * j + 96], msgs[48 * j:48 * j + 48]), j

def test_degenerate_device_mask(gbls, oracle, degen):
    """DeviceMask deltas (k_mask_aggregate over the delta rows, then k_single add / sub) that double, cancel and re-add one key."""
    c = degen.c; n = c.n
    m = gbls.DeviceMask(c.com)
    cur = set()
    def expect():
        assert m.AggregatePublicBytes() == oracle.committee_mask_aggregate(c.och, bitmap_of(n, cur)), sorted(cur)[:12]
    steps = [("bit", 8, True), ("bit", 40, True), ("bit", 104, True), ("bit", 8, False), ("bit", 40, False), ("bit", 104, False),
             ("bit", 5, True), ("bit", 69, True), ("bit", IDENTITY_ROW, True), ("bit", 5, False), ("mask", {8, 40}),
             ("mask", {8, 40, 104, 0, 16}), ("mask", {0, 16, 1, 17}), ("mask", {1, 17}), ("mask", set(range(n))),
             ("mask", set(range(n)) - {8, 40}), ("mask", {5, 69}), ("mask", set())]
    for st in steps:
        if st[0] == "bit":
            m.SetBit(st[1], st[2])
            if st[2]: cur.add(st[1])
            else: cur.discard(st[1])
        else:
            m.SetMask(bitmap_of(n, st[1])); cur = set(st[1])
        expect()

def test_degenerate_signature_sums(gbls, oracle):
    """AggregateSigBytes (k_g2_sum) and BallotBox (k_single G2 add) on equal and opposite signatures."""
    msg = wl.commit_payload("paths/sigsum", 0)
    ks = [wl.seeded_sk("paths/sigsum", i) for i in range(150)]
    sks = b"".join(wl.sk_bytes(k) for k in ks) + b"".join(wl.sk_bytes(R - k) for k in ks)
    sigs, ok = gbls.SignHashBatch(sks, msg * 300, 48)
    assert ok == b"\x01" * 300
    pos = [sigs[96 * i:96 * i + 96] for i in range(150)]; neg = [sigs[96 * (150 + i):96 * (151 + i)] for i in range(150)]
    s, ns = pos[0], neg[0]
    cases = {"s, s": [s, s], "s, -s": [s, ns], "s x 129": [s] * 129, "s x 257": [s] * 257,
             "pairs apart": pos + neg, "pairs adjacent": [x for pr in zip(pos, neg) for x in pr], "pairs apart + s": pos + neg + [s]}
    for name, lst in cases.items():
        assert gbls.AggregateSigBytes(lst) == oracle.aggregate_sigs(lst), name
    assert gbls.AggregateSigBytes([s, ns]) == bytes(96) and gbls.AggregateSigBytes(pos + neg) == bytes(96)
    # ballot box over a 4-key committee: keys 0 and 2 equal, key 1 = -key 0
    blob = gbls.GetPublicKeyBatch(wl.sk_bytes(ks[0]) + wl.sk_bytes(R - ks[0]) + wl.sk_bytes(ks[0]) + wl.sk_bytes(ks[1]))
    com = gbls.Committee([blob[48 * i:48 * i + 48] for i in range(4)])
    one = lambda i: bytes([1 << i])
    box = gbls.BallotBox(com)
    votes = []
    for i, v in ((0, s), (2, s), (1, ns), (3, pos[1])):
        assert box.AddVote(one(i), v) is True
        votes.append(v)
        assert box.Aggregate()[0] == oracle.aggregate_sigs(votes), i
    box2 = gbls.BallotBox(com)
    assert box2.AddVote(one(0), s) and box2.AddVote(one(1), ns)
    assert box2.Aggregate() == (bytes(96), b"\x03")


# ----------------------------------------------------------------------------------------------------------------- E. shapes
SIZES = (1, 7, 8, 9, 32, 33, 128, 129, 511, 512, 513, 700, 1000, 2000)

@pytest.mark.parametrize("n", SIZES)
def test_committee_sizes_warp_kernel(gbls, oracle, orc, n):
    """Committees around the warp width, the 512-entry list limit and beyond, k in {0, 1, n - 1, n, n / 2} signers with the padding
    bits of the last byte set: MaskAggregate bytes and AggregateVerifyBatch booleans (warp kernel) equal the oracle's."""
    sks = [wl.seeded_sk(f"paths/n{n}", i) for i in range(n)]
    c = make_committee(gbls, oracle, sks)
    ks = sorted({k for k in (0, 1, n - 1, n, n // 2) if 0 <= k <= n})
    bms, msgs, sums = [], [], []
    for t, k in enumerate(ks):
        bm = bytearray(wl.bitmap_with_k(f"paths/n{n}", t, n, k))
        if n % 8: bm[-1] |= (0xff << (n % 8)) & 0xff
        bms.append(bytes(bm)); msgs.append(wl.commit_payload(f"paths/n{n}", t)); sums.append(wl.round_signer_sum(sks, bytes(bm)))
    sigs, ok = gbls.SignHashBatch(b"".join(wl.sk_bytes(s) for s in sums), b"".join(msgs), 48)
    sigs = [sigs[96 * t:96 * t + 96] if sums[t] else bytes(96) for t in range(len(ks))]
    for bm in bms:
        assert c.com.MaskAggregate(bm) == oracle.committee_mask_aggregate(c.och, bm)
    # each round twice: as signed, and with a changed message
    B_bm = bms + bms; B_sg = sigs + sigs; B_mm = msgs + [bytes([m[0] ^ 1]) + m[1:] for m in msgs]
    exp = bytes([1 if s else 0 for s in sums] + [0] * len(ks))
    res = c.com.AggregateVerifyBatch(b"".join(B_bm), b"".join(B_sg), b"".join(B_mm), 48)
    assert res == exp, (ks, res)
    for j in range(len(exp)):
        assert (res[j] == 1) == orc.verdict(c.och, B_bm[j], B_sg[j], B_mm[j]), (ks[j % len(ks)], j)

def serial_branch(n, k):
    """The branch k_mask_aggregate_serial takes for k set bits of n."""
    if 2 * k > n and n - k <= HB_MASK_LIST: return "complement"
    return "list" if k <= HB_MASK_LIST else "plain"

@pytest.mark.parametrize("n, ks", [(700, (300, 600, 699, 1, 512, 188)), (2000, (1000, 1100, 900, 1999, 513))])
def test_serial_kernel_branches(gbls, orc, oracle, sm, n, ks):
    """k_mask_aggregate_serial at B = 256 * SM for committees other than 250: n = 700 takes the index list (k <= 512) and the
    complement (n - k <= 512); n = 2000 with k about 1 000 takes the plain loop over every row (row n - 1 always set there)."""
    import numpy as np
    sks = [wl.seeded_sk(f"paths/s{n}", i) for i in range(n)]
    c = make_committee(gbls, oracle, sks)
    bms = []
    for t, k in enumerate(ks):
        bm = bytearray(wl.bitmap_with_k(f"paths/s{n}", t, n, k))
        if serial_branch(n, k) == "plain" and not bm[(n - 1) >> 3] >> ((n - 1) & 7) & 1:     # the plain loop must reach row n - 1
            i = next(i for i in range(n) if bm[i >> 3] >> (i & 7) & 1)
            bm[i >> 3] &= ~(1 << (i & 7)) & 0xff; bm[(n - 1) >> 3] |= 1 << ((n - 1) & 7)
        bms.append(bytes(bm))
    branches = {serial_branch(n, k) for k in ks}
    assert branches == ({"list", "complement"} if n == 700 else {"plain", "complement"}), branches
    agg = [wl.sk_bytes(wl.round_signer_sum(sks, bm)) for bm in bms]
    B = 256 * sm
    nb = len(bms)
    msgs = np.random.default_rng(n).integers(0, 256, B * 48, dtype=np.uint8).tobytes()
    sigs, ok = gbls.SignHashBatch((b"".join(agg) * (B // nb + 1))[:32 * B], msgs, 48)
    assert ok == b"\x01" * B
    pool = SimpleNamespace(c=c, bms=bms, agg=agg, bitmaps=(b"".join(bms) * (B // nb + 1))[:c.blen * B], sigs=sigs, msgs=msgs)
    b = Batch(pool, B).plant(spread(B, extra=(1, 2, 3)), kinds=("wrong_msg", "swapped_sig"))
    r = b.verify(gbls)
    check(orc, b, r, sample=12)
    r1 = Batch(pool, B - 4).verify(gbls)           # no tail on either side: the launch counts differ by the sort kernels
    assert r1.res == b"\x01" * (B - 4)
    assert_other_path(r, r1, "serial | warp mask kernel")

MSG_LENS = (0, 1, 31, 47, 48, 49, 64)

@pytest.mark.parametrize("regime", list(REGIMES))
def test_message_lengths(gbls, orc, pool, regime):
    """msg_len in {0, 1, 31, 47, 48, 49, 64}: bytes beyond 48 do not change the verdict; msg_len 0 (one empty message for every round,
    the same-message form) maps to no point, so every round is 0, as in the oracle."""
    import numpy as np
    B, knobs = REGIMES[regime]
    set_knobs(gbls, **knobs)
    c = pool.c
    reps = B // 16 + 1
    agg = (b"".join(pool.agg) * reps)[:32 * B]
    for L in MSG_LENS:
        rng = np.random.default_rng(1000 + L)
        msgs = bytearray(rng.integers(1, 256, B * L, dtype=np.uint8).tobytes())
        sigs, ok = gbls.SignHashBatch(agg, bytes(msgs), L)
        assert ok == (b"\x01" if L else b"\x00") * B, L
        if L > 48:      # redraw everything past byte 48 after signing
            tail = rng.integers(0, 256, (B, L - 48), dtype=np.uint8)
            for j in range(B): msgs[L * j + 48:L * j + L] = tail[j].tobytes()
        p = SimpleNamespace(c=c, bitmaps=(b"".join(pool.bms) * reps)[:c.blen * B], sigs=sigs, msgs=bytes(msgs))
        b = Batch(p, B, msg_len=L)
        if L:
            b.plant(spread(B, extra=(B // 5,)), kinds=("wrong_msg", "flipped_bitmap_bit", "undecodable_sig"))
        r = b.verify(gbls)
        if not L:
            assert r.res == bytes(B)
            for j in range(0, B, max(1, B // 6)):
                assert not orc.verdict(c.och, *b.round(j))
            continue
        check(orc, b, r, sample=8, seed=L)

def edge_values():
    return {"p-1": P - 1, "p": P, "p+1": P + 1, "2^380": 1 << 380, "2^381-1": (1 << 381) - 1}

def test_edge_message_values(gbls, oracle, orc, pool, defaults):
    """48-byte messages encoding p - 1, p, p + 1, 2^380 and 2^381 - 1 (little-endian; the values >= p are reduced by the 380-bit
    mask of hash_to_fp) verify through every hash-to-G2 form and fail with one byte flipped.  SignHashBatch and MapToG2 give the
    oracle's bytes."""
    c = pool.c
    ev = edge_values()
    emsgs = [v.to_bytes(48, "little") for v in ev.values()]
    for m in emsgs:
        assert gbls.MapToG2(m) == oracle.map_to_g2(m) is not None
    ne = len(emsgs)
    sks = [pool.agg[t % 16] for t in range(ne)]
    sigs, ok = gbls.SignHashBatch(b"".join(sks), b"".join(emsgs), 48)
    assert ok == b"\x01" * ne
    esigs = [oracle.sign_hash(sks[t], emsgs[t]) for t in range(ne)]
    assert sigs == b"".join(esigs)
    # rounds 0 .. ne-1: edge messages; ne .. 2ne-1: the same with byte 0 flipped; then valid pool rounds (24 in all)
    B = 24
    b = Batch(pool, B)
    for t in range(ne):
        for j, m in ((t, emsgs[t]), (ne + t, bytes([emsgs[t][0] ^ 1]) + emsgs[t][1:])):
            b.bm[c.blen * j:c.blen * (j + 1)] = pool.bms[t % 16]; b.sg[96 * j:96 * j + 96] = esigs[t]; b.mm[48 * j:48 * j + 48] = m
        b.bad[ne + t] = "flipped edge message"
    for j in range(B):
        assert (b.expected()[j] == 1) == orc.verdict(c.och, *b.round(j)), j
    forms = [("warp per message", {}), ("warp fall-back", {"hash_fallback": 1}), ("lane pair", {"hash_coop_max": 0}),
             ("k_hash_to_g2", {"mode": 0, "coop_max": 4, "hash_split": 0}), ("map + cofactor", {"mode": 0, "coop_max": 4, "hash_split": 1}),
             ("map + cofactor (Jacobian)", {"mode": 0, "coop_max": 4, "hash_split": 2}),
             ("batched k_hash_to_g2", {"rlc_min": 16, "hash_split": 0}), ("batched map + cofactor", {"rlc_min": 16, "hash_split": 1}),
             ("batched map + cofactor (Jacobian)", {"rlc_min": 16})]
    for name, knobs in forms:
        reset_knobs(gbls, defaults)
        set_knobs(gbls, hm_cache=0, **knobs)
        r = b.verify(gbls)
        assert r.res == b.expected(), (name, r.res)

def encodings():
    out = []
    for name, v in (("p-1", P - 1), ("p", P), ("p+1", P + 1)):
        for flag in (0, 0x80):
            out.append((f"{name}/{flag:#x}", v, flag))
    return out

def test_edge_key_and_signature_encodings(gbls, oracle, triples):
    """Public keys with x = p - 1, p, p + 1 and signatures with x.a or x.b = p - 1, p, p + 1, both sign-flag values: accept / reject of
    every decode kernel equals the oracle's -- k_g1_decode (committee), k_g1_decode_jac (VerifyBatch), k_g2_decode with and without
    the separate subgroup kernel, k_g2_decode_pair, and the AggregateSig decode."""
    pks, sgs = [], []
    for name, v, flag in encodings():
        b = bytearray(v.to_bytes(48, "little")); b[47] |= flag; pks.append((name, bytes(b)))
        for where in ("a", "b", "ab"):
            va = v if "a" in where else 1
            vb = v if "b" in where else 0
            s = bytearray(va.to_bytes(48, "little") + vb.to_bytes(48, "little")); s[95] |= flag
            sgs.append((f"{name}/{where}", bytes(s)))
    for name, pk in pks:
        exp = oracle.pk_check(pk)
        try: gbls.Committee([pk]); got = True
        except ValueError: got = False
        assert got == exp, ("k_g1_decode", name)
    # triples: edge key with a valid signature, valid key with an edge signature; items past the edges are valid
    k0 = 8
    tp = [pk for _, pk in pks] + [triples.pks[48 * i:48 * i + 48] for i in range(len(sgs))] + [triples.pks[48 * i:48 * i + 48] for i in range(k0)]
    ts = [triples.sigs[96 * i:96 * i + 96] for i in range(len(pks))] + [s for _, s in sgs] + [triples.sigs[96 * i:96 * i + 96] for i in range(k0)]
    tm = [triples.msgs[32 * i:32 * i + 32] for i in range(len(pks))] + [triples.msgs[32 * i:32 * i + 32] for i in range(len(sgs))] + [triples.msgs[32 * i:32 * i + 32] for i in range(k0)]
    exp = [None] * len(tp)
    for i in range(len(tp)):
        if not oracle.pk_check(tp[i]): exp[i] = gbls.VB_BAD_KEY_ENCODING
        elif not oracle.sig_check(ts[i]): exp[i] = gbls.VB_BAD_SIG_ENCODING
        else: exp[i] = gbls.VB_OK if oracle.verify_hash(ts[i], tp[i], tm[i]) else gbls.VB_BAD_SIG
    exp = bytes(exp)
    assert exp[-k0:] == bytes([gbls.VB_OK]) * k0
    runs = {}
    for name, knobs in (("k_g2_decode_pair", {}), ("k_g2_decode + k_g2_subgroup", {"coop_max": 0, "mode": 0}),
                        ("k_g2_decode", {"coop_max": 0, "mode": 0, "decode_split": 0})):
        set_knobs(gbls, **knobs)
        runs[name] = call(gbls, lambda: gbls.VerifyBatchStatus(b"".join(tp), b"".join(ts), b"".join(tm), 32))
        assert runs[name].res == exp, (name, [(i, runs[name].res[i], exp[i]) for i in range(len(exp)) if runs[name].res[i] != exp[i]])
    assert_other_path(runs["k_g2_decode_pair"], runs["k_g2_decode + k_g2_subgroup"], "lane-pair | thread decode")
    assert_other_path(runs["k_g2_decode + k_g2_subgroup"], runs["k_g2_decode"], "decode_split 1 | 0")
    for name, s in sgs:
        try: gbls.AggregateSigBytes([s]); got = True
        except ValueError: got = False
        assert got == oracle.sig_check(s), ("k_g2_decode (AggregateSig)", name)
        sig = gbls.Sign()
        try: sig.Deserialize(s); got = True
        except ValueError: got = False
        assert got == oracle.sig_check(s), ("Sign.Deserialize", name)
