"""GPU: concurrent per-call operations (include/hbls.h "Threading").  Python threads call the herumi-shaped API at once (ctypes
releases the GIL), so their requests are coalesced into shared device batches; every caller must still get exactly the oracle's
answer and the bytes of a lone call."""
import ctypes, os, random, subprocess, threading, time
import pytest
from harmony_b200 import workload as wl

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
R_MONT = pow(2, 384, P)
TIMEOUT = 300

# ------------------------------------------------------------------ expected struct bytes of Deserialize: [x R, y R, R] (Montgomery)
def _fp(v): return (v * R_MONT % P).to_bytes(48, "little")
def _f2mul(a, b): return ((a[0] * b[0] - a[1] * b[1]) % P, (a[0] * b[1] + a[1] * b[0]) % P)
def _f2pow(a, e):
    r = (1, 0)
    while e:
        if e & 1: r = _f2mul(r, a)
        a = _f2mul(a, a); e >>= 1
    return r
def _f2sqrt(a):
    """p = 3 mod 4: a^((p-3)/4) route (one square root of a square a, or None)."""
    a1 = _f2pow(a, (P - 3) // 4); alpha = _f2mul(_f2mul(a1, a1), a); x0 = _f2mul(a1, a)
    if alpha == (P - 1, 0): x = ((-x0[1]) % P, x0[0])
    else: x = _f2mul(_f2pow(((1 + alpha[0]) % P, alpha[1]), (P - 1) // 2), x0)
    return x if _f2mul(x, x) == a else None

def g1_struct(enc48):
    v = int.from_bytes(enc48, "little")
    if v == 0: return bytes(144)
    odd = v >> 383; x = v & ((1 << 383) - 1)
    y = pow((x ** 3 + 4) % P, (P + 1) // 4, P)
    if (y & 1) != odd: y = (P - y) % P
    return _fp(x) + _fp(y) + _fp(1)

def g2_struct(enc96):
    a, b = int.from_bytes(enc96[:48], "little"), int.from_bytes(enc96[48:], "little")
    if a == 0 and b == 0: return bytes(288)
    odd = b >> 383; x = (a, b & ((1 << 383) - 1))
    t = _f2mul(_f2mul(x, x), x); y = _f2sqrt(((t[0] + 4) % P, (t[1] + 4) % P))
    if (y[0] & 1) != odd: y = ((-y[0]) % P, (-y[1]) % P)
    return _fp(x[0]) + _fp(x[1]) + _fp(y[0]) + _fp(y[1]) + _fp(1) + _fp(0)

def on_curve_g1(rng):
    while True:
        x = rng.randrange(1, P)
        if pow((x ** 3 + 4) % P, (P - 1) // 2, P) == 1:
            b = bytearray(x.to_bytes(48, "little")); b[47] |= rng.choice([0, 0x80]); return bytes(b)
def on_curve_g2(rng):
    while True:
        x = (rng.randrange(P), rng.randrange(1, P))
        t = _f2mul(_f2mul(x, x), x); t = ((t[0] + 4) % P, (t[1] + 4) % P)
        if pow((t[0] * t[0] + t[1] * t[1]) % P, (P - 1) // 2, P) == 1:
            b = bytearray(x[0].to_bytes(48, "little") + x[1].to_bytes(48, "little")); b[95] |= rng.choice([0, 0x80]); return bytes(b)

# ------------------------------------------------------------------ helpers
def run_threads(n, body):
    """n threads released together by a Barrier; body(t) -> value; returns the values in thread order (raises on a hang)."""
    bar = threading.Barrier(n); out = [None] * n; err = []
    def w(t):
        try:
            bar.wait(); out[t] = body(t)
        except BaseException as e:          # noqa: BLE001 -- reported below
            err.append(e)
    th = [threading.Thread(target=w, args=(t,), daemon=True) for t in range(n)]
    for x in th: x.start()
    for x in th: x.join(TIMEOUT)
    assert not any(x.is_alive() for x in th), "threads still running: deadlock or lost wakeup"
    if err: raise err[0]
    return out

def secret(bls, sk_int):
    s = bls.SecretKey(); s.Deserialize(wl.sk_bytes(sk_int)); return s

def stats(bls):
    return bls.CoalesceStats()

@pytest.fixture(scope="module")
def mat(gbls, oracle):
    """keys, signatures and the oracle's answers for a pool of cases"""
    bls = gbls
    sks = [wl.seeded_sk("conc", i) for i in range(8)]
    pk48 = [oracle.get_public_key(wl.sk_bytes(k)) for k in sks]
    msgs = [wl.commit_payload("conc", j) for j in range(6)] + [wl.seeded_bytes("conc/32", 0, 32)]
    sig96 = {(i, j): oracle.sign_hash(wl.sk_bytes(sks[i]), msgs[j]) for i in range(len(sks)) for j in range(len(msgs))}
    pubs = []
    for p in pk48:
        o = bls.PublicKey(); o.Deserialize(p); pubs.append(o)
    sigs = {}
    for key, s in sig96.items():
        o = bls.Sign(); o.Deserialize(s); sigs[key] = o
    return dict(sks=sks, pk48=pk48, msgs=msgs, sig96=sig96, pubs=pubs, sigs=sigs)

def make_case(rng, bls, oracle, m, t):
    """one mixed call and its expected outcome: (kind, args, expected)"""
    sks, msgs = m["sks"], m["msgs"]
    i, j = rng.randrange(len(sks)), rng.randrange(len(msgs))
    kind = rng.choice(["verify", "verify_msg", "verify_key", "verify_id", "sign_shared", "sign_unique", "sig_des", "pk_des", "getpk"])
    if kind == "verify": return ("verify", (m["sigs"][(i, j)], m["pubs"][i], msgs[j]), True)
    if kind == "verify_msg": return ("verify", (m["sigs"][(i, j)], m["pubs"][i], msgs[(j + 1) % len(msgs)]), False)
    if kind == "verify_key": return ("verify", (m["sigs"][(i, j)], m["pubs"][(i + 1) % len(sks)], msgs[j]), False)
    if kind == "verify_id": return ("verify", (m["sigs"][(i, j)], bls.PublicKey(), msgs[j]), False)
    if kind == "sign_shared": return ("sign", (i, msgs[j]), m["sig96"][(i, j)])
    if kind == "sign_unique":
        msg = wl.seeded_bytes(f"conc/u{t}", rng.randrange(1 << 30), 48)
        return ("sign", (i, msg), oracle.sign_hash(wl.sk_bytes(sks[i]), msg))
    if kind == "sig_des":
        b = rng.choice([m["sig96"][(i, j)], rng.randbytes(96), on_curve_g2(rng), bytes(96)])
        return ("sig_des", (b,), g2_struct(b) if oracle.sig_check(b) else None)
    if kind == "pk_des":
        b = rng.choice([m["pk48"][i], rng.randbytes(48), on_curve_g1(rng), bytes(48)])
        return ("pk_des", (b,), g1_struct(b) if oracle.pk_check(b) else None)
    return ("getpk", (i,), m["pk48"][i])

def do_case(bls, m, sk_objs, case):
    kind, a, _ = case
    if kind == "verify": return a[0].VerifyHash(a[1], a[2])
    if kind == "sign":
        s = sk_objs[a[0]].SignHash(a[1]); return s.Serialize() if s is not None else None
    if kind == "sig_des":
        o = bls.Sign(); ctypes.memset(ctypes.byref(o.v), 0x77, 288)
        n = bls.lib().blsSignatureDeserialize(ctypes.byref(o.v), a[0], 96)
        return bytes(o.v) if n == 96 else (None if bytes(o.v) == b"\x77" * 288 else "touched")
    if kind == "pk_des":
        o = bls.PublicKey(); ctypes.memset(ctypes.byref(o.v), 0x77, 144)
        n = bls.lib().blsPublicKeyDeserialize(ctypes.byref(o.v), a[0], 48)
        return bytes(o.v) if n == 48 else (None if bytes(o.v) == b"\x77" * 144 else "touched")
    return sk_objs[a[0]].GetPublicKey().Serialize()

# ------------------------------------------------------------------ 4. parity under concurrency
def test_mixed_calls_64_threads_match_oracle(gbls, oracle, mat):
    bls = gbls; rng = random.Random(2024)
    sk_objs = [secret(bls, k) for k in mat["sks"]]
    cases = [[make_case(rng, bls, oracle, mat, t) for _ in range(20)] for t in range(64)]
    kinds = {c[0] for row in cases for c in row}
    assert kinds == {"verify", "sign", "sig_des", "pk_des", "getpk"}
    s0 = stats(bls)
    got = run_threads(64, lambda t: [do_case(bls, mat, sk_objs, c) for c in cases[t]])
    s1 = stats(bls)
    for t in range(64):
        for c, g in zip(cases[t], got[t]):
            assert g == c[2], (t, c[0], c[1][:1])
    assert s1["requests"] - s0["requests"] >= 64 * 20
    assert s1["largest_batch"] > 1                                    # 64 threads at once: some calls shared a batch

# ------------------------------------------------------------------ 5. coalescing behind a long batch call
def test_requests_pile_up_behind_a_batch_call(gbls, oracle, mat):
    bls = gbls
    sks = mat["sks"]; pks = mat["pk48"]
    com = bls.Committee(pks)
    B = 16384
    bm = bytes([0xff]) * com.blen()
    msgs = [wl.seeded_bytes("pile", j, 48) for j in range(B)]
    agg = wl.sk_bytes(sum(sks) % wl.R_ORDER)
    sigs, ok = bls.SignHashBatch(agg * B, b"".join(msgs), 48)
    assert ok == b"\x01" * B
    want = [(i % 8, i % 7, i % 3 != 0) for i in range(64)]          # (key, message, valid)
    batch_res = {}
    def long_call():
        batch_res["r"] = com.AggregateVerifyBatch(bm * B, sigs, b"".join(msgs), 48)
    s0 = stats(bls)
    lt = threading.Thread(target=long_call, daemon=True); lt.start()
    time.sleep(0.005)                                                  # the batch call now holds the library mutex
    def one(t):
        i, j, valid = want[t]
        return mat["sigs"][(i, j)].VerifyHash(mat["pubs"][i if valid else (i + 1) % 8], mat["msgs"][j])
    got = run_threads(64, one)
    lt.join(TIMEOUT); assert not lt.is_alive()
    s1 = stats(bls)
    assert got == [v for _, _, v in want]
    assert batch_res["r"] == b"\x01" * B
    assert s1["requests"] - s0["requests"] == 64
    assert s1["batches"] - s0["batches"] <= 2, (s0, s1)

# ------------------------------------------------------------------ 6. lone caller, and the H(m) cache across a coalesced burst
def test_single_thread_runs_batches_of_one_and_burst_fills_hm_cache(gbls, oracle, mat):
    bls = gbls
    sk_objs = [secret(bls, k) for k in mat["sks"]]
    s0 = stats(bls)
    for j in range(5):
        assert mat["sigs"][(1, j)].VerifyHash(mat["pubs"][1], mat["msgs"][j])
        assert sk_objs[2].SignHash(mat["msgs"][j]).Serialize() == mat["sig96"][(2, j)]
        o = bls.Sign(); o.Deserialize(mat["sig96"][(3, j)])
        assert bytes(o.v) == g2_struct(mat["sig96"][(3, j)])
    s1 = stats(bls)
    assert s1["requests"] - s0["requests"] == 15 and s1["batches"] - s0["batches"] == 15
    fresh = [wl.seeded_bytes("burst", j, 48) for j in range(8)]
    sigs = run_threads(64, lambda t: sk_objs[t % 8].SignHash(fresh[t % 8]))
    for t in range(64):
        assert sigs[t].Serialize() == oracle.sign_hash(wl.sk_bytes(mat["sks"][t % 8]), fresh[t % 8])
    h0 = bls.HashCacheStats()
    for t in range(8):
        assert sigs[t].VerifyHash(mat["pubs"][t], fresh[t])
    h1 = bls.HashCacheStats()
    assert h1["hits"] - h0["hits"] == 8 and h1["misses"] == h0["misses"]

# ------------------------------------------------------------------ 7. no deadlock against everything else that takes the mutex
def test_no_deadlock_with_batch_calls_params_committees_and_masks(gbls, oracle, mat):
    bls = gbls
    pks = mat["pk48"]; sks = mat["sks"]
    com = bls.Committee(pks)
    mask = bls.DeviceMask(com)
    B = 64
    bm = bytes([0xff]) * com.blen(); msgs = [wl.seeded_bytes("dl", j, 48) for j in range(B)]
    agg = wl.sk_bytes(sum(sks) % wl.R_ORDER)
    sigs, _ = bls.SignHashBatch(agg * B, b"".join(msgs), 48)
    coop = bls.GetParam("coop_max")
    stop = threading.Event(); errors = []
    def loop(fn):
        def w():
            try:
                while not stop.is_set(): fn()
            except BaseException as e:      # noqa: BLE001
                errors.append(e)
        return w
    def part2(): assert com.AggregateVerifyBatch(bm * B, sigs, b"".join(msgs), 48) == b"\x01" * B
    flip = [0]
    def params(): flip[0] ^= 1; bls.SetParam("coop_max", 64 if flip[0] else coop)
    def committees(): c = bls.Committee(pks[:3]); assert len(c) == 3; del c
    def masks(): mask.SetBit(flip[0] % 8, True); mask.SetBit((flip[0] + 3) % 8, False)
    bg = [threading.Thread(target=loop(f), daemon=True) for f in (part2, params, committees, masks)]
    for x in bg: x.start()
    sk_objs = [secret(bls, k) for k in sks]
    try:
        for rnd in range(3):
            res = run_threads(32, lambda t: (mat["sigs"][(t % 8, rnd)].VerifyHash(mat["pubs"][t % 8], mat["msgs"][rnd]),
                                             sk_objs[t % 8].SignHash(mat["msgs"][rnd]).Serialize()))
            assert all(v and s == mat["sig96"][(t % 8, rnd)] for t, (v, s) in enumerate(res))
    finally:
        stop.set()
        for x in bg: x.join(TIMEOUT)
        bls.SetParam("coop_max", coop)
    assert not any(x.is_alive() for x in bg), "a background caller never returned"
    if errors: raise errors[0]

# ------------------------------------------------------------------ 8. DeviceMask.SetBit from many threads
def test_concurrent_set_bit_keeps_every_bit(gbls, oracle):
    bls = gbls
    n = 40
    pks = [oracle.get_public_key(wl.sk_bytes(wl.seeded_sk("setbit", i))) for i in range(n)]
    com = bls.Committee(pks); mask = bls.DeviceMask(com)
    for rep in range(3):
        mask.Clear()
        run_threads(32, lambda t: mask.SetBit(t, True))
        bm = mask.Mask()
        assert all(bm[i >> 3] >> (i & 7) & 1 for i in range(32)) and mask.CountEnabled() == 32, bm.hex()
        assert mask.AggregatePublicBytes() == com.MaskAggregate(bm) == oracle.mask_aggregate(pks, bm)

# ------------------------------------------------------------------ 9. the same through the C ABI from std::threads (the cgo pattern)
def test_cpp_threads_through_c_abi(gbls, tmp_path):
    from harmony_b200 import build
    exe = str(tmp_path / "hbls_concurrency_test")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-o", exe, os.path.join(ROOT, "harmony_b200", "host", "hbls_concurrency_test.cpp"),
                           "-L" + build.LIBDIR, "-lhbls", "-Wl,-rpath," + build.LIBDIR, "-pthread"])
    r = subprocess.run([exe, "64", "16"], capture_output=True, text=True, timeout=TIMEOUT)
    assert r.returncode == 0 and "all checks passed" in r.stdout, r.stdout + r.stderr
