"""GPU parity tests: the CUDA path, called through the C ABI (ctypes on libhbls.so), against the CPU oracle
(oracle/hbls_oracle.c, pinned to the reference fixtures) and the committed golden vectors.  Bar: bit-exact bytes
and identical booleans.  Restates the reference's functional pins:
  consensus/quorum/quorom_test.go:73-125,381-552  crypto/bls/mask_test.go  consensus/construct_test.go:130-300
"""
import os, random
import pytest
from harmony_b200 import workload as wl

pytestmark = pytest.mark.gpu

P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab

def test_fp_mul_parity(gbls, oracle):
    rng = random.Random(1)
    edge = [0, 1, 2, P - 1, P - 2, (1 << 384) % P, (1 << 380), (1 << 381) - 1 - ((1 << 381) - 1 >= P) * P]
    n = 20000
    vals_a = [rng.randrange(P) for _ in range(n)] + [a for a in edge for _ in edge]
    vals_b = [rng.randrange(P) for _ in range(n)] + [b for _ in edge for b in edge]
    a = b"".join(v.to_bytes(48, "little") for v in vals_a); b = b"".join(v.to_bytes(48, "little") for v in vals_b)
    out = gbls.FpMulBatch(a, b)
    for i, (x, y) in enumerate(zip(vals_a, vals_b)):
        assert int.from_bytes(out[48 * i:48 * i + 48], "little") == x * y % P, (i, hex(x), hex(y))
    # and the C oracle agrees on a sample
    for i in range(0, n, 997):
        assert oracle.fp_mul(a[48 * i:48 * i + 48], b[48 * i:48 * i + 48]) == out[48 * i:48 * i + 48]

def test_golden_sk_to_pk(gbls, fixtures):
    sks = b"".join(bytes.fromhex(v["sk"]) for v in fixtures["sk_pk"])
    pks = gbls.GetPublicKeyBatch(sks)
    for i, v in enumerate(fixtures["sk_pk"]):
        assert pks[48 * i:48 * i + 48].hex() == v["pk"], v["src"]
    # single-op API
    v = fixtures["sk_pk"][0]
    sk = gbls.SecretKey(); sk.DeserializeHexStr(v["sk"])
    assert sk.GetPublicKey().SerializeToHexStr() == v["pk"]
    assert sk.SerializeToHexStr() == v["sk"]

def test_golden_signature(gbls, fixtures):
    sv = fixtures["sig_vectors"][0]
    sk = gbls.SecretKey(); sk.DeserializeHexStr(sv["sk"])
    msg = bytes.fromhex(sv["msg"])
    sig = sk.SignHash(msg)
    assert sig is not None and sig.SerializeToHexStr() == sv["sig"]
    pk = gbls.PublicKey(); pk.DeserializeHexStr(sv["pk"])
    s2 = gbls.Sign(); s2.DeserializeHexStr(sv["sig"])
    assert s2.IsEqual(sig)
    assert s2.VerifyHash(pk, msg)
    assert not s2.VerifyHash(pk, bytes([msg[0] ^ 1]) + msg[1:])
    # staking/types/validator.go:510-532 VerifyBLSKey composition through the batch entry
    assert gbls.VerifyBatch(bytes.fromhex(sv["pk"]), bytes.fromhex(sv["sig"]), msg, 32) == b"\x01"

def test_genesis_pubkeys_decode(gbls, oracle, fixtures):
    pks = [bytes.fromhex(h) for h in fixtures["genesis_pubkeys_sample"][:64]]
    c = gbls.Committee(pks)          # decodes + subgroup-checks all of them on the GPU
    assert len(c) == len(pks)
    for p in pks[:8]:
        assert oracle.pk_check(p)
    bm = bytes([0xff] * ((len(pks) + 7) // 8 - 1) + [(1 << ((len(pks) - 1) % 8 + 1)) - 1])
    assert c.MaskAggregate(bm) == oracle.mask_aggregate(pks, bm)

def test_map_to_g2_parity(gbls, oracle):
    rng = random.Random(7)
    msgs = [b"\x01", bytes(8), rng.randbytes(32), rng.randbytes(48), rng.randbytes(64), b"\xff" * 48, bytes(31) + b"\x01"]
    msgs += [rng.randbytes(rng.choice([1, 8, 32, 40, 48])) for _ in range(24)]
    for m in msgs:
        assert gbls.MapToG2(m) == oracle.map_to_g2(m), m.hex()
    assert gbls.MapToG2(bytes(32)) is None and oracle.map_to_g2(bytes(32)) is None     # t = 0: map undefined
    assert gbls.MapToG2(b"") is None

def test_sign_batch_parity(gbls, oracle):
    n = 40
    sks = [wl.sk_bytes(wl.seeded_sk("t-sign", i)) for i in range(n)]
    msgs = [wl.seeded_bytes("t-sign/m", i, 32) for i in range(n)]
    sigs, ok = gbls.SignHashBatch(b"".join(sks), b"".join(msgs), 32)
    assert ok == b"\x01" * n
    pks = gbls.GetPublicKeyBatch(b"".join(sks))
    for i in range(n):
        assert sigs[96 * i:96 * i + 96] == oracle.sign_hash(sks[i], msgs[i])
        assert pks[48 * i:48 * i + 48] == oracle.get_public_key(sks[i])

def _committee(tag, n):
    sks = [wl.seeded_sk(tag, i) for i in range(n)]
    return sks

def test_config1_four_keys(gbls, oracle):
    """BASELINE configs[0]: 4 keys sign one 32-byte msg, AggregateSig + Verify; bit-exact vs the oracle."""
    sks = _committee("c1", 4)
    msg = wl.seeded_bytes("c1/msg", 0, 32)
    sko = [gbls.SecretKey() for _ in sks]
    for s, k in zip(sko, sks): s.Deserialize(wl.sk_bytes(k))
    pubs = [s.GetPublicKey() for s in sko]
    sigs = [s.SignHash(msg) for s in sko]
    for k, p, s in zip(sks, pubs, sigs):
        assert p.Serialize() == oracle.get_public_key(wl.sk_bytes(k))
        assert s.Serialize() == oracle.sign_hash(wl.sk_bytes(k), msg)
    agg = gbls.AggregateSig(sigs)
    o_agg = oracle.aggregate_sigs([s.Serialize() for s in sigs])
    assert agg.Serialize() == o_agg
    assert gbls.AggregateSigBytes([s.Serialize() for s in sigs]) == o_agg
    wrappers = [gbls.PublicKeyWrapper(p.Serialize(), p) for p in pubs]
    mask = gbls.NewMask(wrappers)
    mask.SetMask(b"\x0f")
    o_apk = oracle.mask_aggregate([w.Bytes for w in wrappers], b"\x0f")
    assert mask.AggregatePublic.Serialize() == o_apk
    assert agg.VerifyHash(mask.AggregatePublic, msg)
    bad = bytes([msg[0] ^ 1]) + msg[1:]
    assert not agg.VerifyHash(mask.AggregatePublic, bad)
    # Sub on 1 -> 0 (mask.go:128-131)
    mask.SetMask(b"\x07")
    assert mask.AggregatePublic.Serialize() == oracle.mask_aggregate([w.Bytes for w in wrappers], b"\x07")
    assert not agg.VerifyHash(mask.AggregatePublic, msg)
    # FastAggregateVerify wrapper == SetMask + VerifyHash
    com = gbls.Committee([w.Bytes for w in wrappers])
    assert gbls.FastAggregateVerify(com, b"\x0f", agg.Serialize(), msg)
    assert not gbls.FastAggregateVerify(com, b"\x07", agg.Serialize(), msg)
    assert oracle.fast_aggregate_verify([w.Bytes for w in wrappers], b"\x0f", o_agg, msg) == 1
    with pytest.raises(ValueError):
        com.AggregateVerify(b"\x0f\x00", agg.Serialize(), msg)

def test_invalid_aggregate_sig_duplicate_signer(gbls):
    """consensus/quorum/quorom_test.go:503-552: an aggregate containing one signer twice fails against the
    de-duplicated key set; the correct set verifies."""
    sks = _committee("dup", 4)
    msg = wl.seeded_bytes("dup/msg", 0, 32)
    sko = []
    for k in sks:
        s = gbls.SecretKey(); s.Deserialize(wl.sk_bytes(k)); sko.append(s)
    pubs = [s.GetPublicKey() for s in sko]
    sigs = [s.SignHash(msg) for s in sko]
    agg_dup = gbls.AggregateSig([sigs[0], sigs[1], sigs[1]])
    agg_ok = gbls.AggregateSig([sigs[0], sigs[1]])
    apk = gbls.PublicKey(); apk.Add(pubs[0]); apk.Add(pubs[1])
    assert not agg_dup.VerifyHash(apk, msg)
    assert agg_ok.VerifyHash(apk, msg)

def test_config2_250_committee_rounds(gbls, oracle):
    """BASELINE configs[1] at test size: 250-validator committee, rounds with k in {167, 200, 250} signers,
    48-byte commit payloads; booleans vs the oracle incl. corrupted rounds."""
    n = 250
    sks = _committee("c2", n)
    pks_blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
    pks = [pks_blob[48 * i:48 * i + 48] for i in range(n)]
    for i in (0, 17, 249):
        assert pks[i] == oracle.get_public_key(wl.sk_bytes(sks[i]))
    com = gbls.Committee(pks)
    och = oracle.committee(pks)
    ks = [167, 200, 250, 167, 200, 250, 1, 249]
    B = len(ks)
    bitmaps = [wl.bitmap_with_k("c2", j, n, ks[j]) for j in range(B)]
    msgs = [wl.commit_payload("c2", j) for j in range(B)]
    agg_sks = [wl.sk_bytes(wl.round_signer_sum(sks, bitmaps[j])) for j in range(B)]
    sigs_blob, ok = gbls.SignHashBatch(b"".join(agg_sks), b"".join(msgs), 48)
    assert ok == b"\x01" * B
    sigs = [sigs_blob[96 * j:96 * j + 96] for j in range(B)]
    assert sigs[0] == oracle.sign_hash(agg_sks[0], msgs[0])
    # mask aggregation bytes
    for j in (0, 2, 6):
        assert com.MaskAggregate(bitmaps[j]) == oracle.committee_mask_aggregate(och, bitmaps[j])
    # corrupt: round 3 wrong message, round 4 bitmap with one extra/missing signer, round 5 signature of another round
    msgs_t = list(msgs); bms_t = list(bitmaps); sigs_t = list(sigs)
    msgs_t[3] = bytes([msgs[3][9] ^ 0x40]).join([msgs[3][:9], msgs[3][10:]])
    b4 = bytearray(bitmaps[4]); b4[0] ^= 1; bms_t[4] = bytes(b4)
    sigs_t[5] = sigs[2]
    res = com.AggregateVerifyBatch(b"".join(bms_t), b"".join(sigs_t), b"".join(msgs_t), 48)
    exp = bytes(1 if oracle.committee_aggregate_verify(och, bms_t[j], sigs_t[j], msgs_t[j]) == 1 else 0 for j in range(B))
    assert res == exp
    assert list(res) == [1, 1, 1, 0, 0, 0, 1, 1]
    # single-round entry
    assert com.AggregateVerify(bitmaps[0], sigs[0], msgs[0]) is True
    assert com.AggregateVerify(bitmaps[0], sigs[1], msgs[0]) is False

def test_individual_sigs_aggregate_250(gbls, oracle):
    """R5: aggregate 250 individually produced signatures on one message; bytes equal oracle and equal the
    signature made with the summed key."""
    n = 250
    sks = _committee("c2", n)
    msg = wl.commit_payload("agg", 0)
    sigs_blob, ok = gbls.SignHashBatch(b"".join(wl.sk_bytes(k) for k in sks), msg * n, 48)
    assert ok == b"\x01" * n
    sigs = [sigs_blob[96 * i:96 * i + 96] for i in range(n)]
    agg = gbls.AggregateSigBytes(sigs)
    assert agg == oracle.aggregate_sigs(sigs)
    assert agg == oracle.sign_hash(wl.sk_bytes(sum(sks) % wl.R_ORDER), msg)
    assert gbls.AggregateSigBytes([]) == bytes(96)

def test_verify_batch_triples(gbls, oracle):
    """BASELINE configs[3] at test size: independent (pk, msg, sig) triples with invalid items at seeded positions."""
    k = 96
    sks = [wl.sk_bytes(wl.seeded_sk("c4", i)) for i in range(k)]
    msgs = [wl.seeded_bytes("c4/m", i, 32) for i in range(k)]
    pks = gbls.GetPublicKeyBatch(b"".join(sks))
    sigs_blob, _ = gbls.SignHashBatch(b"".join(sks), b"".join(msgs), 32)
    sigs = [bytearray(sigs_blob[96 * i:96 * i + 96]) for i in range(k)]
    msgs_t = [bytearray(m) for m in msgs]
    bad = {5: "msg", 17: "sigswap", 40: "sigbyte", 41: "sigbyte", 77: "pkswap"}
    pk_list = [bytearray(pks[48 * i:48 * i + 48]) for i in range(k)]
    for i, kind in bad.items():
        if kind == "msg": msgs_t[i][3] ^= 0x10
        elif kind == "sigswap": sigs[i] = bytearray(sigs_blob[96 * 18:96 * 19])
        elif kind == "sigbyte": sigs[i][10] ^= 0x01
        elif kind == "pkswap": pk_list[i] = bytearray(pks[48 * 78:48 * 79])
    res = gbls.VerifyBatch(b"".join(bytes(p) for p in pk_list), b"".join(bytes(s) for s in sigs), b"".join(bytes(m) for m in msgs_t), 32)
    exp = bytes(1 if oracle.verify_hash(bytes(sigs[i]), bytes(pk_list[i]), bytes(msgs_t[i])) else 0 for i in range(k))
    assert res == exp
    assert all(res[i] == 0 for i in bad) and sum(res) == k - len(bad)

def test_deserialize_rejects(gbls, oracle):
    """Deserialize error behaviour: x >= p, x not on curve, point outside the r-torsion (SURVEY A.5)."""
    pk = gbls.PublicKey()
    with pytest.raises(ValueError): pk.Deserialize(b"\xff" * 48)
    with pytest.raises(ValueError): pk.Deserialize(b"\x00" * 47)
    rng = random.Random(3)
    n_bad = 0
    for _ in range(12):
        b = bytearray(rng.randbytes(48)); b[47] &= 0x99
        exp = oracle.pk_check(bytes(b))
        try: pk.Deserialize(bytes(b)); got = True
        except ValueError: got = False
        assert got == exp; n_bad += (not exp)
    assert n_bad > 0
    sg = gbls.Sign()
    for _ in range(8):
        b = bytearray(rng.randbytes(96)); b[95] &= 0x99; b[47] &= 0x19
        exp = oracle.sig_check(bytes(b))
        try: sg.Deserialize(bytes(b)); got = True
        except ValueError: got = False
        assert got == exp
    # identity encodings round-trip
    pk.Deserialize(bytes(48)); assert pk.Serialize() == bytes(48)
    sg.Deserialize(bytes(96)); assert sg.Serialize() == bytes(96)

def test_mask_semantics(gbls):
    """crypto/bls/mask_test.go: bitmap length errors, SetBit/SetKey/SetKeysAtomic, CountEnabled, policies."""
    sks = _committee("mask", 9)
    wr = []
    for k in sks:
        s = gbls.SecretKey(); s.Deserialize(wl.sk_bytes(k)); wr.append(gbls.WrapperFromPrivateKey(s).Pub)
    m = gbls.NewMask(wr)
    assert m.Len() == 2 and m.CountTotal() == 9 and m.CountEnabled() == 0
    with pytest.raises(ValueError): m.SetMask(b"\x01")
    m.SetBit(0, True); m.SetKey(wr[8].Bytes, True)
    assert m.Mask() == b"\x01\x01" and m.CountEnabled() == 2
    exp = gbls.PublicKey(); exp.Add(wr[0].Object); exp.Add(wr[8].Object)
    assert m.AggregatePublic.IsEqual(exp)
    with pytest.raises(IndexError): m.SetBit(9, True)
    with pytest.raises(KeyError): m.SetKey(b"\x00" * 48, True)
    m.SetKeysAtomic([wr[1], wr[2]], True)
    assert m.IndexEnabled(1) and m.KeyEnabled(wr[2].Bytes) and not m.IndexEnabled(3)
    m.SetBit(0, False); m.SetBit(8, False); m.SetKeysAtomic([wr[1], wr[2]], False)
    assert m.AggregatePublic.Serialize() == bytes(48) and m.CountEnabled() == 0
    assert gbls.NewThresholdPolicy(1).Check(m) is False and gbls.CompletePolicy().Check(m) is False
    m.SetMask(b"\xff\x01"); assert gbls.CompletePolicy().Check(m)
    assert gbls.AggregateMasks(b"\x01\x02", b"\x10\x02") == b"\x11\x02"

def test_string_sign_verify_roundtrip(gbls):
    """Sign(string)/Verify(string): bytes unpinned by the reference (A.7); self-consistent round trip as its tests use it."""
    s = gbls.RandPrivateKey(); p = s.GetPublicKey()
    sig = s.Sign("test message")
    assert sig.Verify(p, "test message") and not sig.Verify(p, "test messagf")

def test_large_batch_properties(gbls):
    """Full-size property check (BASELINE size B=2048 rounds of a 250 committee): all-valid batch verifies, and
    flipping seeded rounds flips exactly those results."""
    n, B = 250, 2048
    sks = _committee("c2", n)
    pks_blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
    com = gbls.Committee([pks_blob[48 * i:48 * i + 48] for i in range(n)])
    # 16 distinct bitmaps/keys reused across rounds keeps host-side generation cheap
    bms = [wl.bitmap_with_k("prop", j, n, [167, 200, 250][j % 3]) for j in range(16)]
    agg = [wl.sk_bytes(wl.round_signer_sum(sks, bm)) for bm in bms]
    msgs = [wl.commit_payload("prop", j) for j in range(B)]
    sigs, ok = gbls.SignHashBatch(b"".join(agg[j % 16] for j in range(B)), b"".join(msgs), 48)
    assert ok == b"\x01" * B
    bitmaps = b"".join(bms[j % 16] for j in range(B))
    res = com.AggregateVerifyBatch(bitmaps, sigs, b"".join(msgs), 48)
    assert res == b"\x01" * B
    rng = random.Random(11); flip = set(rng.sample(range(B), 20))
    msgs2 = [bytes([m[8] ^ 1]).join([m[:8], m[9:]]) if j in flip else m for j, m in enumerate(msgs)]
    res2 = com.AggregateVerifyBatch(bitmaps, sigs, b"".join(msgs2), 48)
    assert all((res2[j] == 0) == (j in flip) for j in range(B))

def test_cpp_host_mirror(gbls):
    """The C++ host mirror (harmony_b200/host/hbls_host.hpp: crypto/bls Mask, multibls, quorum.AggregateVotes,
    chain.verifySignature) restating mask_test.go / quorom_test.go, run as a native binary over libhbls.so."""
    import subprocess
    from harmony_b200 import build
    exe = build.build_host()
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all checks passed" in r.stdout

def test_vrf_roundtrip_and_batch(gbls, oracle):
    """crypto/vrf/bls/bls_vrf_test.go restated: evaluate/verify round trip, truncated proofs and bit flips reject;
    proof bytes equal the oracle's SignHash(sha256(alpha))."""
    import hashlib
    from harmony_b200 import vrf
    sk = gbls.SecretKey(); sk.Deserialize(wl.sk_bytes(wl.seeded_sk("vrf", 0)))
    signer = vrf.NewVRFSigner(sk); verifier = vrf.NewVRFVerifier(sk.GetPublicKey())
    alpha = b"this is a test input"
    beta, pi = signer.Evaluate(alpha)
    assert pi == oracle.sign_hash(wl.sk_bytes(wl.seeded_sk("vrf", 0)), hashlib.sha256(alpha).digest())
    assert beta == hashlib.sha256(pi).digest() and verifier.ProofToHash(alpha, pi) == beta
    with pytest.raises(vrf.ErrInvalidVRF): verifier.ProofToHash(b"other input", pi)
    with pytest.raises(vrf.ErrInvalidVRF): verifier.ProofToHash(alpha, b"")
    with pytest.raises(ValueError): verifier.ProofToHash(alpha, pi[:95])
    bad = bytearray(pi); bad[7] ^= 0x04
    with pytest.raises((ValueError, vrf.ErrInvalidVRF)): verifier.ProofToHash(alpha, bytes(bad))
    pk48 = sk.GetPublicKey().Serialize()
    out = vrf.ProofToHashBatch([pk48] * 4, [alpha, b"x", alpha, alpha], [pi, pi, bytes(bad), pi[:10]])
    assert out[0] == beta and out[1] is None and out[2] is None and out[3] is None

def test_config3_four_shards_and_config5_1000_committee(gbls, oracle):
    """BASELINE configs[2] (4 shards x 250 validators, 4 distinct messages) and configs[4] (1000-validator committee,
    125-byte bitmap) at test size: booleans vs the oracle, one corrupted shard."""
    for n, nshards, tag in ((250, 4, "c3"), (1000, 1, "c5")):
        for sh in range(nshards):
            sks = [wl.seeded_sk(f"{tag}/{sh}", i) for i in range(n)]
            pks_blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
            pks = [pks_blob[48 * i:48 * i + 48] for i in range(n)]
            com = gbls.Committee(pks); och = oracle.committee(pks)
            bm = wl.bitmap_with_k(f"{tag}/{sh}", 0, n, wl.quorum_k(n))
            assert len(bm) == (n + 7) // 8
            msg = wl.commit_payload(f"{tag}/{sh}", 0)
            sig = oracle.sign_hash(wl.sk_bytes(wl.round_signer_sum(sks, bm)), msg)
            if sh == 2: msg = bytes([msg[0] ^ 2]) + msg[1:]
            exp = oracle.committee_aggregate_verify(och, bm, sig, msg) == 1
            assert com.AggregateVerify(bm, sig, msg) == exp == (sh != 2)
            assert com.MaskAggregate(bm) == oracle.committee_mask_aggregate(och, bm)

def test_full_size_batch_serial_mask_and_lockstep_kernels(gbls):
    """BASELINE configs[1] at bench size (37 888 rounds = one full wave): exercises the large-batch kernels
    (complement-based serial mask aggregation, 512-thread lock-stepped lane-pair pairing).  Every honest round verifies;
    rounds whose bitmap gains/loses a signer, or whose payload changes, are exactly the ones rejected."""
    import bench
    n, B = 250, 148 * 256
    sks = bench.make_committee_sks()
    pks_blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
    com = gbls.Committee([pks_blob[48 * i:48 * i + 48] for i in range(n)])
    bitmaps, agg_sk, msgs, nsig = bench.make_rounds(sks, B, seed=7)
    sigs, ok = gbls.SignHashBatch(agg_sk, msgs, 48)
    assert ok == b"\x01" * B
    rng = random.Random(5)
    bad = sorted(rng.sample(range(B), 24))
    bm = bytearray(bitmaps); mm = bytearray(msgs)
    for t, j in enumerate(bad):
        if t % 3 == 0: bm[32 * j + 3] ^= 0x10                  # flip one participation bit (add or remove a signer)
        elif t % 3 == 1: mm[48 * j + 20] ^= 0x01               # different block hash
        else: bm[32 * j + 31] ^= 0x02                          # bit 249: last validator
    sg = bytearray(sigs)
    extra = {100: "x>=p", 2000: "random", 2001: "random", 30000: "identity", 31000: "zero-msg", B - 1: "x>=p"}
    for j, kind in extra.items():
        assert j not in bad
        if kind == "x>=p": sg[96 * j:96 * j + 96] = b"\xff" * 96
        elif kind == "random": sg[96 * j:96 * j + 96] = bytes([(7 * j + 13 * t) & 0xff for t in range(95)] + [0x05])
        elif kind == "identity": sg[96 * j:96 * j + 96] = bytes(96)
        elif kind == "zero-msg": mm[48 * j:48 * j + 48] = bytes(48)
    res = com.AggregateVerifyBatch(bytes(bm), bytes(sg), bytes(mm), 48)
    got = {j for j in range(B) if res[j] != 1}; exp = set(bad) | set(extra)
    assert got == exp, ("unexpected rejects", sorted(got - exp)[:10], "unexpected accepts", sorted(exp - got)[:10], len(got))

def test_leader_vote_collection_same_message(gbls, oracle):
    """R9 (consensus/leader.go:227-290 onCommit loop): 250 validators each send an individual signature on the SAME
    commit payload; the leader verifies every vote.  One device call (bitmap with a single bit per vote, H(m) computed
    once); a multi-key vote (two bits, aggregated signature: leader.go:283 signerPubKey.Add) and two bad votes included."""
    n = 250
    sks = _committee("c2", n)
    pks_blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
    pks = [pks_blob[48 * i:48 * i + 48] for i in range(n)]
    com = gbls.Committee(pks)
    msg = wl.commit_payload("leader", 1)
    sigs_blob, ok = gbls.SignHashBatch(b"".join(wl.sk_bytes(k) for k in sks), msg * n, 48)
    sigs = [bytearray(sigs_blob[96 * i:96 * i + 96]) for i in range(n)]
    bms = []
    for i in range(n):
        bm = bytearray(32); bm[i >> 3] |= 1 << (i & 7); bms.append(bm)
    # vote 7 is a multi-key vote: keys 7 and 8 signed, signatures aggregated by the sender
    sigs[7] = bytearray(oracle.aggregate_sigs([bytes(sigs[7]), bytes(sigs[8])])); bms[7][1] |= 1
    sigs[30] = bytearray(sigs_blob[96 * 31:96 * 32])            # someone else's signature
    bms[99][0] |= 1                                            # claims an extra signer
    res = com.AggregateVerifyBatch(b"".join(bytes(b) for b in bms), b"".join(bytes(s) for s in sigs), msg * n, 48)
    assert [i for i in range(n) if res[i] == 0] == [30, 99]
    assert oracle.verify_hash(bytes(sigs[5]), pks[5], msg) and not oracle.verify_hash(bytes(sigs[30]), pks[30], msg)
    # same votes as independent (pk, msg, sig) triples
    res2 = gbls.VerifyBatch(b"".join(pks[:40]), b"".join(bytes(s) for s in sigs[:40]), msg * 40, 48)
    assert [i for i in range(40) if res2[i] == 0] == [7, 30]    # vote 7 only verifies against pk7 + pk8

def test_batch_mode_rlc_equals_exact(gbls):
    """hbls_set_batch_mode: the random-linear-combination form (groups of 4 rounds, one final exponentiation per group,
    exact fallback) returns the same booleans as the exact per-round form -- on an all-valid batch (no fallback taken), on
    batches with rejected rounds, and for a batch size that leaves a partial group."""
    n = 250
    sks = _committee("c2", n)
    pks_blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
    com = gbls.Committee([pks_blob[48 * i:48 * i + 48] for i in range(n)])
    B = 1024 + 3                                                  # 256 strided groups of 4 + 3 tail rounds
    old_min = gbls.GetParam("rlc_min"); gbls.SetParam("rlc_min", 1024)
    bms = [wl.bitmap_with_k("rlc", j, n, [167, 200, 250][j % 3]) for j in range(16)]
    agg = [wl.sk_bytes(wl.round_signer_sum(sks, bm)) for bm in bms]
    msgs = [wl.commit_payload("rlc", j) for j in range(B)]
    sigs, ok = gbls.SignHashBatch(b"".join(agg[j % 16] for j in range(B)), b"".join(msgs), 48)
    bitmaps = b"".join(bms[j % 16] for j in range(B))
    try:
        for bad in ([], [5], [0, 6, 7, 500, B - 1], [B - 2]):
            m2 = [bytes([m[9] ^ 4]).join([m[:9], m[10:]]) if j in bad else m for j, m in enumerate(msgs)]
            out = {}
            for mode in (1, 0):
                gbls.SetBatchMode(mode)
                out[mode] = com.AggregateVerifyBatch(bitmaps, sigs, b"".join(m2), 48)
            assert out[1] == out[0]
            assert [j for j in range(B) if out[1][j] == 0] == bad
    finally:
        gbls.SetBatchMode(1); gbls.SetParam("rlc_min", old_min)

# ---------------------------------------------------------------------------------------------------------------- round 2
def _bench_committee(gbls):
    import bench
    sks = bench.make_committee_sks()
    pks_blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
    pks = [pks_blob[48 * i:48 * i + 48] for i in range(len(sks))]
    return sks, pks, gbls.Committee(pks)

def test_headline_configuration_rejects_bad_rounds(gbls, oracle):
    """The benchmark's own configuration -- B = 303 104 rounds = 37 888 strided groups of 8 (one chunk of the two-kernel pairing
    k_rlc_lines_split<8> / k_rlc_accum_split<8> in 512-thread lock-stepped persistent CTAs; the fused k_rlc_pairing_split<8> only runs
    with rlc_two_phase 0, see tests/test_gpu_paths.py) -- with >= 30 seeded bad rounds of seven kinds.  Per-round booleans equal the oracle's on every
    bad round and on a 2 000-round random sample; hbls_last_batch_info shows that the G = 8 kernel itself rejected exactly the
    groups that hold a bad round, and that only their rounds went through the exact pass."""
    import bench
    n, B = 250, 303104
    sks, pks, com = _bench_committee(gbls)
    bitmaps, agg_sk, msgs, nsig = bench.make_rounds(sks, B, seed=2025)
    sigs, ok = gbls.SignHashBatch(agg_sk, msgs, 48)
    assert ok == b"\x01" * B
    rng = random.Random(77)
    bad = sorted(rng.sample(range(B), 35))
    bm = bytearray(bitmaps); mm = bytearray(msgs); sg = bytearray(sigs)
    kinds = {}
    for t, j in enumerate(bad):
        kind = ["wrong_msg", "swapped_sig", "flipped_bitmap_bit", "undecodable_sig", "identity_sig", "empty_bitmap", "zero_msg"][t % 7]
        kinds[j] = kind
        if kind == "wrong_msg": mm[48 * j + 17] ^= 0x20
        elif kind == "swapped_sig":
            o = (j + 1) % B; sg[96 * j:96 * j + 96] = sigs[96 * o:96 * o + 96]
        elif kind == "flipped_bitmap_bit": bm[32 * j + (t % 31)] ^= 0x04
        elif kind == "undecodable_sig": sg[96 * j:96 * j + 96] = b"\xff" * 96
        elif kind == "identity_sig": sg[96 * j:96 * j + 96] = bytes(96)
        elif kind == "empty_bitmap": bm[32 * j:32 * j + 32] = bytes(32)
        elif kind == "zero_msg": mm[48 * j:48 * j + 48] = bytes(48)
    res = com.AggregateVerifyBatch(bytes(bm), bytes(sg), bytes(mm), 48)
    info = gbls.LastBatchInfo()
    assert info["mode"] == 1 and info["group_size"] == 8 and info["cta_threads"] == 512 and info["groups"] == B // 8 and info["tail_rounds"] == 0
    ng = B // 8
    bad_groups = {j % ng for j in bad}
    assert info["groups_failed"] == len(bad_groups) and info["rounds_rechecked"] == 8 * len(bad_groups)
    och = oracle.committee(pks)
    check = set(bad) | set(rng.sample(range(B), 2000)) | {g + k * ng for g in list(bad_groups)[:8] for k in range(8)}
    for j in sorted(check):
        exp = oracle.committee_aggregate_verify(och, bytes(bm[32 * j:32 * j + 32]), bytes(sg[96 * j:96 * j + 96]), bytes(mm[48 * j:48 * j + 48])) == 1
        assert (res[j] == 1) == exp, (j, kinds.get(j), res[j])
    assert all(res[j] == 0 for j in bad)
    assert sum(res) == B - len(bad)
    # an all-valid batch of the same size: nothing fails, nothing is re-verified
    res2 = com.AggregateVerifyBatch(bitmaps, sigs, msgs, 48)
    info2 = gbls.LastBatchInfo()
    assert res2 == b"\x01" * B and info2["groups_failed"] == 0 and info2["rounds_rechecked"] == 0

def test_rlc_groups_of_eight_forced_small(gbls, oracle):
    """G = 8 forced at a small batch (hbls_set_param rlc_g / rlc_min): bad, undecodable and identity rounds in several positions
    of the strided groups, a partial tail; booleans equal the exact mode's and the oracle's."""
    n = 250
    sks, pks, com = _bench_committee(gbls)
    och = oracle.committee(pks)
    B = 8 * 9 + 5
    bms = [wl.bitmap_with_k("g8", j, n, [167, 200, 250][j % 3]) for j in range(B)]
    msgs = [wl.commit_payload("g8", j) for j in range(B)]
    sigs_blob, ok = gbls.SignHashBatch(b"".join(wl.sk_bytes(wl.round_signer_sum(sks, bm)) for bm in bms), b"".join(msgs), 48)
    sigs = [bytearray(sigs_blob[96 * j:96 * j + 96]) for j in range(B)]
    msgs = [bytearray(m) for m in msgs]; bms = [bytearray(b) for b in bms]
    msgs[0][3] ^= 1                      # group 0, position 0
    sigs[9 + 4] = bytearray(b"\xff" * 96)  # group 4, position 1: undecodable
    sigs[7 * 9 + 8] = bytearray(96)      # group 8, position 7: identity signature
    bms[3 * 9 + 2] = bytearray(32)       # group 2, position 3: empty bitmap -> identity key
    msgs[B - 1][40] ^= 2                 # tail round
    old = (gbls.GetParam("rlc_g"), gbls.GetParam("rlc_min"))
    try:
        gbls.SetParam("rlc_g", 8); gbls.SetParam("rlc_min", 16)
        out = {}
        for mode in (1, 0):
            gbls.SetBatchMode(mode)
            out[mode] = com.AggregateVerifyBatch(b"".join(bytes(b) for b in bms), b"".join(bytes(s) for s in sigs), b"".join(bytes(m) for m in msgs), 48)
            if mode == 1:
                info = gbls.LastBatchInfo()
                assert info["mode"] == 1 and info["group_size"] == 8 and info["groups"] == 9 and info["tail_rounds"] == 5
                assert info["groups_failed"] == 4 and info["rounds_rechecked"] == 32
        exp = bytes(1 if oracle.committee_aggregate_verify(och, bytes(bms[j]), bytes(sigs[j]), bytes(msgs[j])) == 1 else 0 for j in range(B))
        assert out[1] == out[0] == exp
        assert [j for j in range(B) if exp[j] == 0] == [0, 13, 29, 71, B - 1]
    finally:
        gbls.SetBatchMode(1); gbls.SetParam("rlc_g", old[0]); gbls.SetParam("rlc_min", old[1])

def test_config4_ten_thousand_triples_one_percent_invalid(gbls, oracle):
    """BASELINE configs[3] at full size on one GPU: 10 000 independent (pk, msg, sig) triples from 10 000 distinct keys, 1 % invalid
    (bit-flipped signature byte, wrong message, wrong key, undecodable key) at seeded positions.  Goes through the batched groups
    (triple form: P_j = -s_j pk_j) with the exact pass over failed groups; 10 000 booleans equal the oracle's on every invalid item,
    every item that shares a group with one, and a random sample."""
    k = 10000
    sks = b"".join(wl.sk_bytes(wl.seeded_sk("c4full", i)) for i in range(k))
    msgs = b"".join(wl.seeded_bytes("c4full/m", i, 32) for i in range(k))
    pks = gbls.GetPublicKeyBatch(sks)
    sigs, ok = gbls.SignHashBatch(sks, msgs, 32)
    assert ok == b"\x01" * k
    rng = random.Random(404)
    bad = sorted(rng.sample(range(k), 100))
    pk = bytearray(pks); sg = bytearray(sigs); mm = bytearray(msgs)
    for t, i in enumerate(bad):
        kind = t % 4
        if kind == 0: sg[96 * i + 11] ^= 0x01
        elif kind == 1: mm[32 * i + 5] ^= 0x80
        elif kind == 2: o = (i + 7) % k; pk[48 * i:48 * i + 48] = pks[48 * o:48 * o + 48]
        else: pk[48 * i:48 * i + 48] = b"\xff" * 48
    old = gbls.GetParam("rlc_min")
    try:
        gbls.SetParam("rlc_min", 1024)               # batched groups (the default threshold is higher: below it the exact forms are faster)
        res = gbls.VerifyBatch(bytes(pk), bytes(sg), bytes(mm), 32)
        info = gbls.LastBatchInfo()
    finally: gbls.SetParam("rlc_min", old)
    assert info["mode"] == 1 and info["group_size"] == 4 and info["groups"] == k // 4
    # default thresholds decide the form of the second call; forcing the exact warp-per-item path must agree
    assert gbls.VerifyBatch(bytes(pk), bytes(sg), bytes(mm), 32) == res and gbls.LastBatchInfo()["mode"] == (1 if k >= old else 0)
    old_c = gbls.GetParam("coop_max")
    try:
        gbls.SetParam("rlc_min", 1 << 30); gbls.SetParam("coop_max", 1 << 30)
        assert gbls.VerifyBatch(bytes(pk), bytes(sg), bytes(mm), 32) == res and gbls.LastBatchInfo()["cta_threads"] == 32      # warp per item
    finally: gbls.SetParam("rlc_min", old); gbls.SetParam("coop_max", old_c)
    ng = k // 4
    check = set(bad) | {g % ng + q * ng for g in bad for q in range(4)} | set(rng.sample(range(k), 300))
    for i in sorted(check):
        exp = oracle.verify_hash(bytes(sg[96 * i:96 * i + 96]), bytes(pk[48 * i:48 * i + 48]), bytes(mm[32 * i:32 * i + 32]))
        assert (res[i] == 1) == exp, i
    assert all(res[i] == 0 for i in bad) and sum(res) == k - len(bad)
    gbls.SetBatchMode(0)
    try: assert gbls.VerifyBatch(bytes(pk), bytes(sg), bytes(mm), 32) == res
    finally: gbls.SetBatchMode(1)

def test_config3_four_committees_one_call(gbls, oracle):
    """BASELINE configs[2]: 4 shards x 250 validators, 4 distinct messages, ONE device call (hbls_aggregate_verify_items);
    then with shard 2 corrupted, and a 64-item multi-committee batch through the batched groups."""
    n = 250
    coms, ochs, bms, sigs, msgs, skss = [], [], [], [], [], []
    for sh in range(4):
        sks = [wl.seeded_sk(f"c3i/{sh}", i) for i in range(n)]
        blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
        pks = [blob[48 * i:48 * i + 48] for i in range(n)]
        coms.append(gbls.Committee(pks)); ochs.append(oracle.committee(pks)); skss.append(sks)
        bm = wl.bitmap_with_k(f"c3i/{sh}", 0, n, [167, 200, 250, 180][sh]); bms.append(bm)
        m = wl.commit_payload(f"c3i/{sh}", 0); msgs.append(m)
        sigs.append(oracle.sign_hash(wl.sk_bytes(wl.round_signer_sum(sks, bm)), m))
    assert gbls.AggregateVerifyItems(coms, bms, b"".join(sigs), b"".join(msgs), 48) == b"\x01\x01\x01\x01"
    m2 = list(msgs); m2[2] = bytes([m2[2][0] ^ 4]) + m2[2][1:]
    res = gbls.AggregateVerifyItems(coms, bms, b"".join(sigs), b"".join(m2), 48)
    exp = bytes(1 if oracle.committee_aggregate_verify(ochs[j], bms[j], sigs[j], m2[j]) == 1 else 0 for j in range(4))
    assert res == exp == b"\x01\x01\x00\x01"
    # 64 items cycling over the 4 committees, two bad, through the batched groups (rlc_min lowered)
    K = 64; items = [j % 4 for j in range(K)]
    ibm = [wl.bitmap_with_k(f"c3i/b{j}", j, n, 167 + j) for j in range(K)]
    imsg = [wl.commit_payload("c3i/m", j) for j in range(K)]
    isig = [oracle.sign_hash(wl.sk_bytes(wl.round_signer_sum(skss[items[j]], ibm[j])), imsg[j]) for j in range(K)]
    isig[5] = isig[6]; imsg[40] = bytes([imsg[40][9] ^ 1]).join([imsg[40][:9], imsg[40][10:]])
    old = gbls.GetParam("rlc_min")
    try:
        gbls.SetParam("rlc_min", 16)
        res = gbls.AggregateVerifyItems([coms[s] for s in items], ibm, b"".join(isig), b"".join(imsg), 48)
        assert gbls.LastBatchInfo()["mode"] == 1
    finally: gbls.SetParam("rlc_min", old)
    exp = bytes(1 if oracle.committee_aggregate_verify(ochs[items[j]], ibm[j], isig[j], imsg[j]) == 1 else 0 for j in range(K))
    assert res == exp and [j for j in range(K) if res[j] == 0] == [5, 40]

def test_verify_headers_range(gbls, oracle):
    """SURVEY 8f.1 (stagedstreamsync/sig_verify.go:23-58, engine.go:619-642): a block range of one committee epoch in one call.
    Mixed valid / wrong payload / below quorum / quorum reached only through padding bits / undecodable signature; statuses follow
    the reference's order of checks."""
    n = 250
    sks, pks, com = _bench_committee(gbls)
    och = oracle.committee(pks)
    N = 40; q = wl.quorum_k(n)
    bms = [bytearray(wl.bitmap_with_k("hdr", j, n, [167, 200, 250][j % 3])) for j in range(N)]
    msgs = [bytearray(wl.commit_payload("hdr", j)) for j in range(N)]
    sig_blob, ok = gbls.SignHashBatch(b"".join(wl.sk_bytes(wl.round_signer_sum(sks, bytes(b))) for b in bms), b"".join(bytes(m) for m in msgs), 48)
    sigs = [bytearray(sig_blob[96 * j:96 * j + 96]) for j in range(N)]
    msgs[3][12] ^= 1                                                    # wrong payload
    bms[7] = bytearray(wl.bitmap_with_k("hdr/low", 7, n, 160))            # 160 < 167 signers, correctly signed
    sigs[7] = bytearray(oracle.sign_hash(wl.sk_bytes(wl.round_signer_sum(sks, bytes(bms[7]))), bytes(msgs[7])))
    bms[11] = bytearray(wl.bitmap_with_k("hdr/pad", 11, n, 161))          # 161 real signers + the 6 padding bits of byte 31 = 167 raw bits
    sigs[11] = bytearray(oracle.sign_hash(wl.sk_bytes(wl.round_signer_sum(sks, bytes(bms[11]))), bytes(msgs[11])))
    bms[11][31] |= 0xfc
    sigs[20] = bytearray(b"\xff" * 96)                                   # undecodable
    sigs[21] = bytearray(b"\xff" * 96); bms[21] = bytearray(wl.bitmap_with_k("hdr/low", 21, n, 10))   # undecodable AND below quorum: decode error first
    st = com.VerifyHeaders(b"".join(bytes(s) for s in sigs), b"".join(bytes(b) for b in bms), b"".join(bytes(m) for m in msgs), 48, q)
    exp = []
    for j in range(N):
        if not oracle.sig_check(bytes(sigs[j])): exp.append(gbls.HDR_BAD_ENCODING); continue
        cnt = sum(1 for i in range(n) if bms[j][i >> 3] >> (i & 7) & 1)
        if cnt < q: exp.append(gbls.HDR_NO_QUORUM); continue
        exp.append(gbls.HDR_OK if oracle.committee_aggregate_verify(och, bytes(bms[j]), bytes(sigs[j]), bytes(msgs[j])) == 1 else gbls.HDR_BAD_SIG)
    assert list(st) == exp
    assert st[3] == gbls.HDR_BAD_SIG and st[7] == gbls.HDR_NO_QUORUM and st[11] == gbls.HDR_NO_QUORUM and st[20] == st[21] == gbls.HDR_BAD_ENCODING
    assert sum(1 for s in st if s == gbls.HDR_OK) == N - 5
    # quorum = 0 skips the gate (staked-vote deciders apply their own): the correctly signed low-participation header verifies
    st0 = com.VerifyHeaders(b"".join(bytes(s) for s in sigs), b"".join(bytes(b) for b in bms), b"".join(bytes(m) for m in msgs), 48, 0)
    assert st0[7] == gbls.HDR_OK and st0[11] == gbls.HDR_OK and st0[3] == gbls.HDR_BAD_SIG

def test_persistent_device_mask_and_ballot_box(gbls, oracle):
    """SURVEY 8f.2: device-resident Mask (delta Add/Sub like mask.go:121-133,137-155) and running vote aggregate
    (quorum.go:164-196 with each vote decoded once).  Bytes equal the oracle's from-scratch results."""
    n = 250
    sks, pks, com = _bench_committee(gbls)
    och = oracle.committee(pks)
    m = gbls.DeviceMask(com)
    assert m.AggregatePublicBytes() == bytes(48) and m.CountEnabled() == 0
    with pytest.raises(ValueError): m.SetMask(b"\x01")
    with pytest.raises(IndexError): m.SetBit(250, True)
    b1 = wl.bitmap_with_k("dm", 1, n, 200); b2 = wl.bitmap_with_k("dm", 2, n, 170)
    m.SetMask(b1); assert m.AggregatePublicBytes() == oracle.committee_mask_aggregate(och, b1) and m.CountEnabled() == 200
    m.SetMask(b2); assert m.AggregatePublicBytes() == oracle.committee_mask_aggregate(och, b2) and m.Mask() == b2     # mixed Add / Sub delta
    extra = next(i for i in range(n) if not b2[i >> 3] >> (i & 7) & 1)
    m.SetBit(extra, True); b3 = bytearray(b2); b3[extra >> 3] |= 1 << (extra & 7)
    assert m.AggregatePublicBytes() == oracle.committee_mask_aggregate(och, bytes(b3)) and m.CountEnabled() == 171
    m.SetBit(extra, True); assert m.CountEnabled() == 171                   # idempotent: no second Add
    m.SetBit(extra, False); assert m.AggregatePublicBytes() == oracle.committee_mask_aggregate(och, b2)
    pad = bytearray(b2); pad[31] |= 0xfc; m.SetMask(bytes(pad))               # padding bits are ignored (mask.go:121 ranges over Publics)
    assert m.Mask() == b2 and m.CountEnabled() == 170
    msg = wl.commit_payload("dm", 9)
    sig = oracle.sign_hash(wl.sk_bytes(wl.round_signer_sum(sks, b2)), msg)
    assert m.VerifyHash(sig, msg) and not m.VerifyHash(sig, bytes([msg[0] ^ 1]) + msg[1:]) and not m.VerifyHash(b"\xff" * 96, msg)
    m.Clear(); assert m.AggregatePublicBytes() == bytes(48) and not m.VerifyHash(bytes(96), msg)      # identity key never verifies
    # ballot box
    box = gbls.BallotBox(com)
    vmsg = wl.commit_payload("box", 0)
    vs, _ = gbls.SignHashBatch(b"".join(wl.sk_bytes(k) for k in sks[:12]), vmsg * 12, 48)
    one = lambda i: bytes(bytearray((1 << (i & 7)) if b == i >> 3 else 0 for b in range(32)))
    for i in range(10): assert box.AddVote(one(i), vs[96 * i:96 * i + 96]) is True
    assert box.AddVote(one(3), vs[96 * 3:96 * 4]) is False                    # signer 3 already collected
    multi = bytearray(32); multi[1] |= 0x0c                                   # keys 10 and 11 in one multi-key vote
    assert box.AddVote(bytes(multi), oracle.aggregate_sigs([vs[96 * 10:96 * 11], vs[96 * 11:96 * 12]])) is True
    with pytest.raises(ValueError): box.AddVote(one(20), b"\xff" * 96)
    agg, bm = box.Aggregate()
    assert agg == oracle.aggregate_sigs([vs[96 * i:96 * i + 96] for i in range(12)]) and bm == bytes([0xff, 0x0f] + [0] * 30)
    assert com.AggregateVerify(bm, agg, vmsg)

def test_get_address_and_identity_key(gbls, oracle):
    import hashlib
    sk = gbls.SecretKey(); sk.Deserialize(wl.sk_bytes(wl.seeded_sk("addr", 0)))
    pk = sk.GetPublicKey()
    assert pk.GetAddress() == hashlib.sha256(pk.Serialize()).digest()[:20]
    # identity operands (include/hbls.h): zero key + zero signature is NOT a valid signature of anything
    z_pk, z_sig = gbls.PublicKey(), gbls.Sign()
    assert not z_sig.VerifyHash(z_pk, b"\x01" * 32) and not oracle.verify_hash(bytes(96), bytes(48), b"\x01" * 32)
    assert gbls.VerifyBatch(bytes(48), bytes(96), b"\x01" * 32, 32) == b"\x00"
    assert gbls.LastError()[0] == 0

def test_device_entry_on_two_streams(gbls):
    """hbls_aggregate_verify_batch_device is asynchronous on the caller's stream; scratch is per stream, so two pipelines in flight
    on different streams do not clobber each other's intermediates (one batch all valid, the other with rejected rounds)."""
    import torch
    n = 250
    sks, pks, com = _bench_committee(gbls)
    B = 2048
    L = gbls.lib()
    def mk(tag, bad):
        bms = [wl.bitmap_with_k(tag, j % 8, n, [167, 200, 250][j % 3]) for j in range(8)]
        agg = [wl.sk_bytes(wl.round_signer_sum(sks, bm)) for bm in bms]
        msgs = [wl.commit_payload(tag, j) for j in range(B)]
        sigs, ok = gbls.SignHashBatch(b"".join(agg[j % 8] for j in range(B)), b"".join(msgs), 48)
        msgs = [bytes([m[8] ^ 1]).join([m[:8], m[9:]]) if j in bad else m for j, m in enumerate(msgs)]
        dev = lambda b: torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
        return dev(b"".join(bms[j % 8] for j in range(B))), dev(sigs), dev(b"".join(msgs)), torch.full((B,), 7, dtype=torch.uint8, device="cuda")
    bad = {5, 900, 2047}
    A, Bt = mk("s0", set()), mk("s1", bad)
    s0, s1 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    for _ in range(3):
        for (bm, sg, ms, rs), st in ((A, s0), (Bt, s1)):
            rc = L.hbls_aggregate_verify_batch_device(com.h, B, bm.data_ptr(), 32, sg.data_ptr(), ms.data_ptr(), 48, rs.data_ptr(), st.cuda_stream)
            assert rc == 0
    torch.cuda.synchronize()
    assert A[3].cpu().numpy().tobytes() == b"\x01" * B
    r = Bt[3].cpu().numpy().tobytes()
    assert {j for j in range(B) if r[j] == 0} == bad

def test_split_batch_partial_records_fold(gbls, oracle):
    """SURVEY 8e / BASELINE configs[3]: ONE batch split over ranks.  Two slices processed one after the other on this GPU stand for
    two ranks: their 872-byte partial records { sum r sigma, product of Miller values } fold to "all valid" exactly when every triple
    of both slices verifies; a wrong message, a swapped key or an undecodable signature in either slice makes the fold fail, and the
    single-rank protocol (shard.verify_triples_split) then returns the exact per-item booleans."""
    from harmony_b200 import shard
    k = 96
    sks = b"".join(wl.sk_bytes(wl.seeded_sk("split", i)) for i in range(k))
    msgs = b"".join(wl.seeded_bytes("split/m", i, 32) for i in range(k))
    pks = gbls.GetPublicKeyBatch(sks)
    sigs, ok = gbls.SignHashBatch(sks, msgs, 32)
    cut = 41
    def recs(p, s, m): return [gbls.RlcPartial(p[:48 * cut], s[:96 * cut], m[:32 * cut], 32), gbls.RlcPartial(p[48 * cut:], s[96 * cut:], m[32 * cut:], 32)]
    r = recs(pks, sigs, msgs)
    assert all(len(x) == gbls.PARTIAL_BYTES for x in r)
    assert gbls.RlcFold(r) is True and gbls.RlcFold([r[0]]) is True and gbls.RlcFold([r[1]]) is True
    assert gbls.RlcFold(recs(pks, sigs, msgs)) is True                                 # fresh coefficients every call
    m2 = bytearray(msgs); m2[32 * 70 + 3] ^= 1
    assert gbls.RlcFold(recs(pks, sigs, bytes(m2))) is False
    p2 = bytearray(pks); p2[48 * 5:48 * 6] = pks[48 * 6:48 * 7]
    assert gbls.RlcFold(recs(bytes(p2), sigs, msgs)) is False
    s2 = bytearray(sigs); s2[96 * 90:96 * 91] = b"\xff" * 96
    assert gbls.RlcFold(recs(pks, bytes(s2), msgs)) is False
    # errors that cancel under EQUAL coefficients do not cancel here: swap two signatures (sum of signatures unchanged)
    s3 = bytearray(sigs); s3[96 * 10:96 * 11], s3[96 * 11:96 * 12] = sigs[96 * 11:96 * 12], sigs[96 * 10:96 * 11]
    assert gbls.RlcFold(recs(pks, bytes(s3), msgs)) is False
    # the protocol on one rank
    res, settled = shard.verify_triples_split(pks, sigs, msgs, 32)
    assert res == b"\x01" * k and settled is True
    res, settled = shard.verify_triples_split(pks, bytes(s3), bytes(m2), 32)
    assert settled is False and [i for i in range(k) if res[i] == 0] == [10, 11, 70]
    assert res == bytes(1 if oracle.verify_hash(bytes(s3[96 * i:96 * i + 96]), pks[48 * i:48 * i + 48], bytes(m2[32 * i:32 * i + 32])) else 0 for i in range(k))

def test_hash_cache_sign_then_verify(gbls, oracle):
    """H(m) cache (include/hbls.h): the validator signs a block hash / commit payload and later verifies the aggregate over the same
    bytes (consensus/validator.go:219-236).  Cached and uncached paths give the oracle's bytes / booleans; a hit never leaks to
    another message; > 48-byte inputs share the entry of their 48-byte prefix (A.3 truncation); eviction keeps results exact."""
    n = 16
    sks = [wl.seeded_sk("hmc", i) for i in range(n)]
    pks_blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
    pks = [pks_blob[48 * i:48 * i + 48] for i in range(n)]
    com = gbls.Committee(pks); och = oracle.committee(pks)
    bm = wl.bitmap_with_k("hmc", 0, n, 11)
    agg = wl.sk_bytes(wl.round_signer_sum(sks, bm))
    m1 = wl.commit_payload("hmc", 1); m2 = wl.commit_payload("hmc", 2)
    old = gbls.GetParam("hm_cache")
    try:
        gbls.SetParam("hm_cache", 0)
        sk = gbls.SecretKey(); sk.Deserialize(agg)
        cold_sig = sk.SignHash(m1).Serialize()
        assert cold_sig == oracle.sign_hash(agg, m1)
        cold = com.AggregateVerify(bm, cold_sig, m1)
        gbls.SetParam("hm_cache", 1)
        st0 = gbls.HashCacheStats()
        warm_sig = sk.SignHash(m1).Serialize()                       # miss: fills the entry
        assert warm_sig == cold_sig
        assert com.AggregateVerify(bm, warm_sig, m1) == cold == True      # hit
        assert com.AggregateVerify(bm, warm_sig, m2) is False             # other message: miss, rejected
        assert com.AggregateVerify(bm, warm_sig, m2) is False             # ... and rejected again from the cache
        st1 = gbls.HashCacheStats()
        assert st1["hits"] - st0["hits"] == 2 and st1["misses"] - st0["misses"] == 2
        # truncation: 60-byte input = its first 48 bytes
        long_msg = m1 + b"\x55" * 12
        assert sk.SignHash(long_msg).Serialize() == cold_sig
        assert gbls.HashCacheStats()["hits"] - st1["hits"] == 1
        # prefetch, then 70 more distinct messages evict it; every check still exact
        gbls.HashPrefetch(m2)
        sig2 = sk.SignHash(m2).Serialize()
        assert sig2 == oracle.sign_hash(agg, m2)
        for t in range(70): gbls.HashPrefetch(wl.commit_payload("hmc/evict", t))
        assert com.AggregateVerify(bm, sig2, m2) is True and com.AggregateVerify(bm, sig2, m1) is False
        assert oracle.committee_aggregate_verify(och, bm, sig2, m2) == 1
        # same-message vote batch (leader): H(m) from the cache, booleans unchanged
        votes, ok = gbls.SignHashBatch(b"".join(wl.sk_bytes(k) for k in sks), m1 * n, 48)
        sb = b"".join(bytes([1 << (i & 7) if j == i >> 3 else 0 for j in range(2)]) for i in range(n))
        bad = bytearray(votes); bad[96 * 5 + 3] ^= 1
        r1 = com.AggregateVerifyBatch(sb, bytes(bad), m1 * n, 48)
        gbls.SetParam("hm_cache", 0)
        assert com.AggregateVerifyBatch(sb, bytes(bad), m1 * n, 48) == r1 and sum(r1) == n - 1 and r1[5] == 0
    finally:
        gbls.SetParam("hm_cache", old)

def test_hash_paths_agree(gbls, oracle):
    """The small-batch hash-to-G2 forms: lane pair per item, warp per message with the cofactor clearing on the VM, and that kernel's
    fall-back for degenerate group-law cases (forced here).  All give the oracle's bytes through SignHash, and the same verdicts through
    a 40-round batch.  The thread-per-item forms of large batches (hash_split 0 / 1 / 2) are run by tests/test_gpu_paths.py."""
    n = 8
    sks = [wl.seeded_sk("hp", i) for i in range(n)]
    pks_blob = gbls.GetPublicKeyBatch(b"".join(wl.sk_bytes(k) for k in sks))
    com = gbls.Committee([pks_blob[48 * i:48 * i + 48] for i in range(n)])
    B = 40
    bms = [wl.bitmap_with_k("hp", j, n, 6 + (j % 3)) for j in range(B)]
    msgs = [wl.commit_payload("hp", j) for j in range(B)]
    agg = [wl.sk_bytes(wl.round_signer_sum(sks, bm)) for bm in bms]
    sigs, ok = gbls.SignHashBatch(b"".join(agg), b"".join(msgs), 48)
    assert ok == b"\x01" * B and sigs[:96] == oracle.sign_hash(agg[0], msgs[0])
    bad = bytearray(b"".join(msgs)); bad[48 * 7] ^= 1
    names = ("hm_cache", "hash_coop_max", "hash_fallback", "hash_split")
    old = {k: gbls.GetParam(k) for k in names}
    res = {}
    try:
        gbls.SetParam("hm_cache", 0)
        for tag, coop_max, fb in (("warp+vm", 592, 0), ("warp+fallback", 592, 1), ("lane pair", 0, 0)):
            gbls.SetParam("hash_coop_max", coop_max); gbls.SetParam("hash_fallback", fb)
            sk = gbls.SecretKey(); sk.Deserialize(agg[3])
            assert sk.SignHash(msgs[3]).Serialize() == sigs[96 * 3:96 * 4] == oracle.sign_hash(agg[3], msgs[3]), tag
            res[tag] = com.AggregateVerifyBatch(b"".join(bms), sigs, bytes(bad), 48)
        assert res["warp+vm"] == res["warp+fallback"] == res["lane pair"] and res["lane pair"][7] == 0 and sum(res["lane pair"]) == B - 1
    finally:
        for k, v in old.items(): gbls.SetParam(k, v)
