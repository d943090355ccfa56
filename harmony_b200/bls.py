"""harmony_b200/bls.py -- ctypes binding of libhbls.so (include/hbls.h) with the reference's Go names.

Mirrors, identifier for identifier, what Harmony code calls on this path:
  github.com/harmony-one/bls/ffi/go/bls : Init, SecretKey, PublicKey, Sign (SURVEY.md 8b)
  crypto/bls                            : Mask (mask.go:67-242), AggregateSig (mask.go:58-64),
                                          BytesToBLSPublicKey + LRU (mask.go:35-55), SeparateSigAndMask (bls.go:120-136)
plus the BASELINE.json names FastAggregateVerify / VerifyAggregateSig as wrappers over
SetMask + VerifyHash (internal/chain/engine.go:630-640).

Every group / field operation goes through the C ABI into CUDA kernels.  No CPU fallback: if the shared library
or a CUDA device is missing this module raises.
"""
import ctypes, os
from collections import OrderedDict

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("HBLS_LIB") or os.path.join(_HERE, "lib", "libhbls.so")

BLS12_381 = 5
_COMPILED_TIME_VAR = 46
PublicKeySizeInBytes = 48
BLSSignatureSizeInBytes = 96

ERR_CUDA, ERR_ARG, ERR_DECODE = -100, -2, -3

_lib = None
_inited = False

class HblsError(RuntimeError):
    pass

class BatchInfo(ctypes.Structure):
    """hbls_batch_info (include/hbls.h)."""
    _fields_ = [("mode", ctypes.c_int32), ("group_size", ctypes.c_int32), ("rounds", ctypes.c_uint64), ("groups", ctypes.c_uint64),
                ("groups_failed", ctypes.c_uint32), ("rounds_rechecked", ctypes.c_uint32), ("tail_rounds", ctypes.c_uint32),
                ("cta_threads", ctypes.c_uint32)]
    def as_dict(self): return {k: int(getattr(self, k)) for k, _ in self._fields_}

class _Sec(ctypes.Structure):
    _fields_ = [("d", ctypes.c_uint64 * 4)]
class _Pub(ctypes.Structure):
    _fields_ = [("d", ctypes.c_uint64 * 18)]
class _Sig(ctypes.Structure):
    _fields_ = [("d", ctypes.c_uint64 * 36)]

def lib():
    """Load libhbls.so (built in-tree by harmony_b200/build.py); raise loudly when absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise HblsError(f"{_LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(the BLS backend is CUDA-only; there is no CPU fallback)")
        L = ctypes.CDLL(_LIB_PATH)
        c = ctypes
        vp, sz, u8p = c.c_void_p, c.c_size_t, c.c_char_p
        def sig(name, res, *args):
            f = getattr(L, name); f.restype = res; f.argtypes = list(args)
        sig("blsInit", c.c_int, c.c_int, c.c_int)
        sig("hbls_init_device", c.c_int, c.c_int)
        sig("blsSecretKeySetByCSPRNG", c.c_int, c.POINTER(_Sec))
        sig("blsGetPublicKey", None, c.POINTER(_Pub), c.POINTER(_Sec))
        sig("blsSignHash", c.c_int, c.POINTER(_Sig), c.POINTER(_Sec), u8p, sz)
        sig("blsVerifyHash", c.c_int, c.POINTER(_Sig), c.POINTER(_Pub), u8p, sz)
        sig("blsSign", None, c.POINTER(_Sig), c.POINTER(_Sec), u8p, sz)
        sig("blsVerify", c.c_int, c.POINTER(_Sig), c.POINTER(_Pub), u8p, sz)
        sig("blsPublicKeyAdd", None, c.POINTER(_Pub), c.POINTER(_Pub))
        sig("blsPublicKeySub", None, c.POINTER(_Pub), c.POINTER(_Pub))
        sig("blsSignatureAdd", None, c.POINTER(_Sig), c.POINTER(_Sig))
        sig("blsSecretKeySerialize", sz, vp, sz, c.POINTER(_Sec))
        sig("blsPublicKeySerialize", sz, vp, sz, c.POINTER(_Pub))
        sig("blsSignatureSerialize", sz, vp, sz, c.POINTER(_Sig))
        sig("blsSecretKeyDeserialize", sz, c.POINTER(_Sec), u8p, sz)
        sig("blsPublicKeyDeserialize", sz, c.POINTER(_Pub), u8p, sz)
        sig("blsSignatureDeserialize", sz, c.POINTER(_Sig), u8p, sz)
        sig("blsSecretKeyIsEqual", c.c_int, c.POINTER(_Sec), c.POINTER(_Sec))
        sig("blsPublicKeyIsEqual", c.c_int, c.POINTER(_Pub), c.POINTER(_Pub))
        sig("blsSignatureIsEqual", c.c_int, c.POINTER(_Sig), c.POINTER(_Sig))
        sig("hbls_committee_create", c.c_int, c.POINTER(vp), u8p, sz, c.POINTER(sz))
        sig("hbls_committee_destroy", None, vp)
        sig("hbls_committee_size", sz, vp)
        sig("hbls_mask_aggregate", c.c_int, vp, u8p, sz, vp)
        sig("hbls_aggregate_sigs", c.c_int, u8p, sz, vp)
        sig("hbls_aggregate_verify", c.c_int, vp, u8p, sz, u8p, u8p, sz)
        sig("hbls_aggregate_verify_batch", c.c_int, vp, sz, vp, sz, vp, vp, sz, vp)
        sig("hbls_aggregate_verify_batch_device", c.c_int, vp, sz, vp, sz, vp, vp, sz, vp, vp)
        sig("hbls_verify_batch", c.c_int, sz, vp, vp, vp, sz, vp)
        sig("hbls_verify_batch_status", c.c_int, sz, vp, vp, vp, sz, vp)
        sig("hbls_sign_hash_batch", c.c_int, sz, vp, vp, sz, vp, vp)
        sig("hbls_get_public_key_batch", c.c_int, sz, vp, vp)
        sig("hbls_map_to_g2", c.c_int, u8p, sz, vp)
        sig("hbls_fp_mul_batch", c.c_int, sz, vp, vp, vp)
        sig("hbls_kernel_launch_count", c.c_uint64)
        sig("hbls_build_info", c.c_int)
        sig("hbls_probe_mac32_per_s", c.c_double, c.c_int, c.POINTER(c.c_double))
        sig("hbls_get_address", c.c_int, c.POINTER(_Pub), vp)
        sig("hbls_last_error", c.c_int, vp, sz)
        sig("hbls_last_batch_info", c.c_int, c.POINTER(BatchInfo))
        sig("hbls_set_param", c.c_int, u8p, c.c_longlong)
        sig("hbls_get_param", c.c_longlong, u8p)
        sig("hbls_aggregate_verify_items", c.c_int, sz, c.POINTER(vp), vp, vp, vp, sz, vp)
        sig("hbls_verify_headers", c.c_int, vp, sz, vp, vp, sz, vp, sz, sz, vp)
        sig("hbls_rlc_partial", c.c_int, sz, vp, vp, vp, sz, vp)
        sig("hbls_rlc_fold", c.c_int, sz, vp)
        sig("hbls_mask_create", c.c_int, c.POINTER(vp), vp)
        sig("hbls_mask_destroy", None, vp)
        sig("hbls_mask_set_mask", c.c_int, vp, vp, sz)
        sig("hbls_mask_set_bit", c.c_int, vp, sz, c.c_int)
        sig("hbls_mask_clear", c.c_int, vp)
        sig("hbls_mask_count_enabled", c.c_int, vp)
        sig("hbls_mask_get", c.c_int, vp, vp, sz, vp)
        sig("hbls_mask_verify", c.c_int, vp, u8p, u8p, sz)
        sig("hbls_ballot_box_create", c.c_int, c.POINTER(vp), vp)
        sig("hbls_ballot_box_destroy", None, vp)
        sig("hbls_ballot_box_add_vote", c.c_int, vp, u8p, sz, u8p)
        sig("hbls_ballot_box_aggregate", c.c_int, vp, vp, vp, sz)
        sig("hbls_selftest_split", c.c_int, c.c_uint32)
        sig("hbls_set_batch_mode", None, c.c_int)
        sig("hbls_get_batch_mode", c.c_int)
        sig("hbls_hash_prefetch", c.c_int, u8p, sz)
        sig("hbls_hash_cache_stats", c.c_int, c.POINTER(c.c_uint64), c.POINTER(c.c_uint64))
        sig("hbls_coalesce_stats", c.c_int, c.POINTER(c.c_uint64), c.POINTER(c.c_uint64), c.POINTER(c.c_uint64))
        sig("hbls_stage_timing_enable", None, c.c_int)
        sig("hbls_stage_timing_get", c.c_int, c.POINTER(c.c_float), c.c_int)
        _lib = L
    return _lib

def Init(curve=BLS12_381, device=None):
    """bls.Init(bls.BLS12_381) (crypto/bls/mask.go:18-20).  Raises when no CUDA device is usable."""
    global _inited
    L = lib()
    rc = L.hbls_init_device(device) if device is not None else L.blsInit(curve, _COMPILED_TIME_VAR)
    if rc != 0:
        raise HblsError(f"blsInit failed rc={rc}: a CUDA device is required (no CPU fallback)")
    _inited = True

def _need():
    if not _inited:
        Init()
    return _lib

def _buf(b):
    return bytes(b)

# ------------------------------------------------------------------ ffi/go/bls value types
class SecretKey:
    def __init__(self): self.v = _Sec()
    def SetByCSPRNG(self):
        if _need().blsSecretKeySetByCSPRNG(ctypes.byref(self.v)) != 0: raise HblsError("SetByCSPRNG failed")
    def GetPublicKey(self):
        pk = PublicKey(); _need().blsGetPublicKey(ctypes.byref(pk.v), ctypes.byref(self.v)); return pk
    def SignHash(self, h: bytes):
        """nil (None) on failure, like the Go wrapper (callers check != nil: consensus/construct.go:101)."""
        s = Sign()
        return s if _need().blsSignHash(ctypes.byref(s.v), ctypes.byref(self.v), _buf(h), len(h)) == 0 else None
    def Sign(self, m):
        m = m.encode() if isinstance(m, str) else m
        s = Sign(); _need().blsSign(ctypes.byref(s.v), ctypes.byref(self.v), _buf(m), len(m)); return s
    def Serialize(self) -> bytes:
        out = ctypes.create_string_buffer(32); n = _need().blsSecretKeySerialize(out, 32, ctypes.byref(self.v)); return out.raw[:n]
    def Deserialize(self, b: bytes):
        if _need().blsSecretKeyDeserialize(ctypes.byref(self.v), _buf(b), len(b)) == 0: raise ValueError("err blsSecretKeyDeserialize")
    def SerializeToHexStr(self): return self.Serialize().hex()
    def DeserializeHexStr(self, s: str): self.Deserialize(bytes.fromhex(s))
    def IsEqual(self, o): return _need().blsSecretKeyIsEqual(ctypes.byref(self.v), ctypes.byref(o.v)) == 1

class PublicKey:
    """Zero value = identity (crypto/bls/mask.go:88).  Plain value type: copy() is a struct copy."""
    def __init__(self): self.v = _Pub()
    def copy(self):
        p = PublicKey(); ctypes.memmove(ctypes.byref(p.v), ctypes.byref(self.v), ctypes.sizeof(_Pub)); return p
    def Serialize(self) -> bytes:
        out = ctypes.create_string_buffer(48); n = _need().blsPublicKeySerialize(out, 48, ctypes.byref(self.v)); return out.raw[:n]
    def Deserialize(self, b: bytes):
        if _need().blsPublicKeyDeserialize(ctypes.byref(self.v), _buf(b), len(b)) == 0: raise ValueError("err blsPublicKeyDeserialize")
    def SerializeToHexStr(self): return self.Serialize().hex()
    def DeserializeHexStr(self, s: str): self.Deserialize(bytes.fromhex(s))
    def Add(self, rhs): _need().blsPublicKeyAdd(ctypes.byref(self.v), ctypes.byref(rhs.v))
    def Sub(self, rhs): _need().blsPublicKeySub(ctypes.byref(self.v), ctypes.byref(rhs.v))
    def IsEqual(self, o): return _need().blsPublicKeyIsEqual(ctypes.byref(self.v), ctypes.byref(o.v)) == 1
    def GetAddress(self) -> bytes:
        """[20]byte (internal/utils/utils.go:77): first 20 bytes of SHA-256(Serialize())."""
        out = ctypes.create_string_buffer(20)
        if _need().hbls_get_address(ctypes.byref(self.v), out) != 0: raise HblsError("hbls_get_address failed")
        return out.raw

class Sign:
    """Zero value = identity (crypto/bls/mask.go:59)."""
    def __init__(self): self.v = _Sig()
    def copy(self):
        p = Sign(); ctypes.memmove(ctypes.byref(p.v), ctypes.byref(self.v), ctypes.sizeof(_Sig)); return p
    def Serialize(self) -> bytes:
        out = ctypes.create_string_buffer(96); n = _need().blsSignatureSerialize(out, 96, ctypes.byref(self.v)); return out.raw[:n]
    def Deserialize(self, b: bytes):
        if _need().blsSignatureDeserialize(ctypes.byref(self.v), _buf(b), len(b)) == 0: raise ValueError("err blsSignatureDeserialize")
    def SerializeToHexStr(self): return self.Serialize().hex()
    def DeserializeHexStr(self, s: str): self.Deserialize(bytes.fromhex(s))
    def Add(self, rhs): _need().blsSignatureAdd(ctypes.byref(self.v), ctypes.byref(rhs.v))
    def VerifyHash(self, pub: PublicKey, h: bytes) -> bool:
        return _need().blsVerifyHash(ctypes.byref(self.v), ctypes.byref(pub.v), _buf(h), len(h)) == 1
    def Verify(self, pub: PublicKey, m) -> bool:
        m = m.encode() if isinstance(m, str) else m
        return _need().blsVerify(ctypes.byref(self.v), ctypes.byref(pub.v), _buf(m), len(m)) == 1
    def IsEqual(self, o): return _need().blsSignatureIsEqual(ctypes.byref(self.v), ctypes.byref(o.v)) == 1

# ------------------------------------------------------------------ crypto/bls (bls.go, mask.go)
class PublicKeyWrapper:
    """crypto/bls/bls.go:30-33: serialized + deserialized form."""
    def __init__(self, bytes_: bytes, obj: PublicKey): self.Bytes = bytes(bytes_); self.Object = obj
    def Hex(self): return self.Bytes.hex()

class PrivateKeyWrapper:
    def __init__(self, pri: SecretKey, pub: PublicKeyWrapper): self.Pri = pri; self.Pub = pub

def WrapperFromPrivateKey(pri: SecretKey) -> PrivateKeyWrapper:
    pub = pri.GetPublicKey()
    return PrivateKeyWrapper(pri, PublicKeyWrapper(pub.Serialize(), pub))

def RandPrivateKey() -> SecretKey:
    s = SecretKey(); s.SetByCSPRNG(); return s

_BLS_PUBKEY_CACHE_SIZE = 1024
BLSPubKeyCache = OrderedDict()

def BytesToBLSPublicKey(b: bytes) -> PublicKey:
    """crypto/bls/mask.go:35-55 incl. the 1024-entry LRU keyed by the raw bytes."""
    if len(b) == 0: raise ValueError("BytesToBLSPublicKey: empty input")
    k = bytes(b)
    if k in BLSPubKeyCache:
        BLSPubKeyCache.move_to_end(k); return BLSPubKeyCache[k].copy()
    pk = PublicKey(); pk.Deserialize(k)
    BLSPubKeyCache[k] = pk.copy()
    if len(BLSPubKeyCache) > _BLS_PUBKEY_CACHE_SIZE: BLSPubKeyCache.popitem(last=False)
    return pk

def AggregateSig(sigs) -> Sign:
    """crypto/bls/mask.go:58-64: fold Sign.Add from the zero value."""
    agg = Sign()
    for s in sigs: agg.Add(s)
    return agg

def SeparateSigAndMask(commit_sigs: bytes):
    """crypto/bls/bls.go:120-136."""
    if len(commit_sigs) < BLSSignatureSizeInBytes:
        raise ValueError("no mask data found in commit sigs")
    return bytes(commit_sigs[:96]), bytes(commit_sigs[96:])

class Committee:
    """Device-resident decoded public-key table (hbls_committee_*): the GPU analogue of the epochCtx cache of
    internal/chain/engine.go:644-659.  Keys are decoded and subgroup-checked once, on the GPU."""
    def __init__(self, pubkeys48):
        L = _need()
        blob = b"".join(bytes(p) for p in pubkeys48)
        self.n = len(blob) // 48
        self.h = ctypes.c_void_p()
        bad = ctypes.c_size_t(0)
        rc = L.hbls_committee_create(ctypes.byref(self.h), blob, self.n, ctypes.byref(bad))
        if rc == ERR_DECODE: raise ValueError(f"invalid public key at index {bad.value}")
        if rc != 0: raise HblsError(f"hbls_committee_create rc={rc}")
    def __del__(self):
        try:
            if self.h and _lib is not None: _lib.hbls_committee_destroy(self.h); self.h = None
        except Exception: pass
    def __len__(self): return self.n
    def blen(self): return (self.n + 7) >> 3
    def MaskAggregate(self, bitmap: bytes) -> bytes:
        out = ctypes.create_string_buffer(48)
        rc = _lib.hbls_mask_aggregate(self.h, _buf(bitmap), len(bitmap), out)
        if rc == ERR_ARG: raise ValueError(f"mismatching bitmap lengths expectedBitmapLength {self.blen()} providedBitmapLength {len(bitmap)}")
        if rc != 0: raise HblsError(f"hbls_mask_aggregate rc={rc}")
        return out.raw
    def AggregateVerify(self, bitmap: bytes, sig96: bytes, msg: bytes) -> bool:
        rc = _lib.hbls_aggregate_verify(self.h, _buf(bitmap), len(bitmap), _buf(sig96), _buf(msg), len(msg))
        if rc == ERR_ARG: raise ValueError(f"mismatching bitmap lengths expectedBitmapLength {self.blen()} providedBitmapLength {len(bitmap)}")
        if rc < 0: raise HblsError(f"hbls_aggregate_verify rc={rc}")
        return rc == 1
    def AggregateVerifyBatch(self, bitmaps: bytes, sigs96: bytes, msgs: bytes, msg_len: int) -> bytes:
        B = len(sigs96) // 96
        assert len(bitmaps) == B * self.blen() and len(msgs) == B * msg_len
        res = ctypes.create_string_buffer(B if B else 1)
        rc = _lib.hbls_aggregate_verify_batch(self.h, B, _buf(bitmaps), self.blen(), _buf(sigs96), _buf(msgs), msg_len, res)
        if rc != 0: raise HblsError(f"hbls_aggregate_verify_batch rc={rc}")
        return res.raw[:B]

    def VerifyHeaders(self, sigs96: bytes, bitmaps: bytes, payloads: bytes, payload_len: int, quorum: int) -> bytes:
        """Block-range form of engine.go:619-642 verifySignature: one status byte per header (HDR_* below)."""
        n = len(sigs96) // 96
        assert len(bitmaps) == n * self.blen() and len(payloads) == n * payload_len
        st = ctypes.create_string_buffer(n if n else 1)
        rc = _lib.hbls_verify_headers(self.h, n, _buf(sigs96), _buf(bitmaps), self.blen(), _buf(payloads), payload_len, quorum, st)
        if rc != 0: raise HblsError(f"hbls_verify_headers rc={rc}")
        return st.raw[:n]

HDR_BAD_SIG, HDR_OK, HDR_NO_QUORUM, HDR_BAD_ENCODING = 0, 1, 2, 3

def AggregateVerifyItems(committees, bitmaps, sigs96: bytes, msgs: bytes, msg_len: int) -> bytes:
    """Multi-committee batch (BASELINE configs[2]; crosslinks engine.go:592-604): item j = (committees[j], bitmaps[j], sig_j, msg_j)."""
    k = len(committees)
    arr = (ctypes.c_void_p * k)(*[c.h for c in committees])
    blob = b"".join(bytes(b) for b in bitmaps)
    res = ctypes.create_string_buffer(k if k else 1)
    rc = _need().hbls_aggregate_verify_items(k, arr, _buf(blob), _buf(sigs96), _buf(msgs), msg_len, res)
    if rc == ERR_ARG: raise ValueError("hbls_aggregate_verify_items: bad argument")
    if rc != 0: raise HblsError(f"hbls_aggregate_verify_items rc={rc}")
    return res.raw[:k]

def FastAggregateVerify(committee: Committee, bitmap: bytes, sig96: bytes, msg: bytes) -> bool:
    """BASELINE.json name; == Deserialize + Mask.SetMask + aggSig.VerifyHash(mask.AggregatePublic, msg)
    (internal/chain/engine.go:630-640)."""
    return committee.AggregateVerify(bitmap, sig96, msg)
VerifyAggregateSig = FastAggregateVerify

def AggregateSigBytes(sigs96) -> bytes:
    """AggregateSig on serialized signatures (consensus/quorum/quorum.go:164-196 re-decodes hex ballots)."""
    blob = b"".join(bytes(s) for s in sigs96)
    out = ctypes.create_string_buffer(96)
    rc = _need().hbls_aggregate_sigs(blob, len(blob) // 96, out)
    if rc == ERR_DECODE: raise ValueError("err blsSignatureDeserialize")
    if rc != 0: raise HblsError(f"hbls_aggregate_sigs rc={rc}")
    return out.raw

def VerifyBatch(pks48: bytes, sigs96: bytes, msgs: bytes, msg_len: int) -> bytes:
    k = len(sigs96) // 96
    res = ctypes.create_string_buffer(k if k else 1)
    rc = _need().hbls_verify_batch(k, _buf(pks48), _buf(sigs96), _buf(msgs), msg_len, res)
    if rc != 0: raise HblsError(f"hbls_verify_batch rc={rc}")
    return res.raw[:k]

VB_BAD_SIG, VB_OK, VB_BAD_SIG_ENCODING, VB_BAD_KEY_ENCODING = 0, 1, 3, 4
def VerifyBatchStatus(pks48: bytes, sigs96: bytes, msgs: bytes, msg_len: int) -> bytes:
    """hbls_verify_batch_status: one VB_* byte per triple -- which of BytesToBLSPublicKey / Sign.Deserialize / VerifyHash failed,
    in the order the reference meets them (consensus/view_change_msg.go:139-190, consensus/checks.go:20-39)."""
    k = len(sigs96) // 96
    st = ctypes.create_string_buffer(k if k else 1)
    rc = _need().hbls_verify_batch_status(k, _buf(pks48), _buf(sigs96), _buf(msgs), msg_len, st)
    if rc != 0: raise HblsError(f"hbls_verify_batch_status rc={rc}")
    return st.raw[:k]

PARTIAL_BYTES = 872
def RlcPartial(pks48: bytes, sigs96: bytes, msgs: bytes, msg_len: int) -> bytes:
    """Partial record of a slice of triples (hbls_rlc_partial): what a rank contributes to the all-gather of a batch split over GPUs."""
    k = len(sigs96) // 96
    rec = ctypes.create_string_buffer(PARTIAL_BYTES)
    rc = _need().hbls_rlc_partial(k, _buf(pks48), _buf(sigs96), _buf(msgs), msg_len, rec)
    if rc != 0: raise HblsError(f"hbls_rlc_partial rc={rc}")
    return rec.raw
def RlcFold(records) -> bool:
    """True iff the gathered records prove every item of every slice valid (hbls_rlc_fold)."""
    blob = b"".join(bytes(r) for r in records)
    rc = _need().hbls_rlc_fold(len(blob) // PARTIAL_BYTES, _buf(blob))
    if rc < 0: raise HblsError(f"hbls_rlc_fold rc={rc}")
    return rc == 1

def SignHashBatch(sks32: bytes, msgs: bytes, msg_len: int):
    k = len(sks32) // 32
    out = ctypes.create_string_buffer(96 * k if k else 1); ok = ctypes.create_string_buffer(k if k else 1)
    rc = _need().hbls_sign_hash_batch(k, _buf(sks32), _buf(msgs), msg_len, out, ok)
    if rc != 0: raise HblsError(f"hbls_sign_hash_batch rc={rc}")
    return out.raw[:96 * k], ok.raw[:k]

def HashPrefetch(msg: bytes):
    """Enqueue H(msg) into the library's device-resident H(m) cache and return at once (include/hbls.h: e.g. on ANNOUNCE, when the
    block hash / commit payload the node will sign and later verify becomes known)."""
    rc = _need().hbls_hash_prefetch(_buf(msg), len(msg))
    if rc != 0: raise HblsError(f"hbls_hash_prefetch rc={rc}")

def HashCacheStats():
    h = ctypes.c_uint64(0); m = ctypes.c_uint64(0)
    _need().hbls_hash_cache_stats(ctypes.byref(h), ctypes.byref(m))
    return {"hits": h.value, "misses": m.value}

def CoalesceStats():
    """Coalescing of concurrent per-call operations (VerifyHash, SignHash, Deserialize, GetPublicKey) since the library was loaded:
    requests queued, batches run, largest batch.  ctypes releases the GIL around each call, so Python threads coalesce too."""
    r = ctypes.c_uint64(0); b = ctypes.c_uint64(0); m = ctypes.c_uint64(0)
    _need().hbls_coalesce_stats(ctypes.byref(r), ctypes.byref(b), ctypes.byref(m))
    return {"requests": r.value, "batches": b.value, "largest_batch": m.value}

def GetPublicKeyBatch(sks32: bytes) -> bytes:
    k = len(sks32) // 32
    out = ctypes.create_string_buffer(48 * k if k else 1)
    rc = _need().hbls_get_public_key_batch(k, _buf(sks32), out)
    if rc != 0: raise HblsError(f"hbls_get_public_key_batch rc={rc}")
    return out.raw[:48 * k]

def MapToG2(msg: bytes):
    out = ctypes.create_string_buffer(96)
    rc = _need().hbls_map_to_g2(_buf(msg), len(msg), out)
    return out.raw if rc == 0 else None

def FpMulBatch(a48: bytes, b48: bytes) -> bytes:
    n = len(a48) // 48
    out = ctypes.create_string_buffer(48 * n if n else 1)
    rc = _need().hbls_fp_mul_batch(n, _buf(a48), _buf(b48), out)
    if rc != 0: raise HblsError(f"hbls_fp_mul_batch rc={rc}")
    return out.raw[:48 * n]

class Mask:
    """crypto/bls/mask.go:67-242 -- participation bitmap + running aggregate public key (Add on 0->1, Sub on 1->0)."""
    def __init__(self, publics):
        self.Publics = list(publics)
        self.PublicsIndex = {p.Bytes: i for i, p in enumerate(self.Publics)}
        self.Bitmap = bytearray(self.Len())
        self.AggregatePublic = PublicKey()
    def Clear(self):
        self.Bitmap = bytearray(self.Len()); self.AggregatePublic = PublicKey()
    def Mask(self): return bytes(self.Bitmap)
    def Len(self): return (len(self.Publics) + 7) >> 3
    def SetMask(self, mask: bytes):
        if self.Len() != len(mask):
            raise ValueError(f"mismatching bitmap lengths expectedBitmapLength {self.Len()} providedBitmapLength {len(mask)}")
        for i in range(len(self.Publics)):
            byt, msk = i >> 3, 1 << (i & 7)
            if (self.Bitmap[byt] & msk) == 0 and (mask[byt] & msk) != 0:
                self.Bitmap[byt] ^= msk; self.AggregatePublic.Add(self.Publics[i].Object)
            if (self.Bitmap[byt] & msk) != 0 and (mask[byt] & msk) == 0:
                self.Bitmap[byt] ^= msk; self.AggregatePublic.Sub(self.Publics[i].Object)
    def SetBit(self, i: int, enable: bool):
        if i >= len(self.Publics): raise IndexError("index out of range")
        byt, msk = i >> 3, 1 << (i & 7)
        if (self.Bitmap[byt] & msk) == 0 and enable:
            self.Bitmap[byt] ^= msk; self.AggregatePublic.Add(self.Publics[i].Object)
        if (self.Bitmap[byt] & msk) != 0 and not enable:
            self.Bitmap[byt] ^= msk; self.AggregatePublic.Sub(self.Publics[i].Object)
    def GetPubKeyFromMask(self, flag: bool):
        return [p.Object for i, p in enumerate(self.Publics) if bool(self.Bitmap[i >> 3] & (1 << (i & 7))) == flag]
    def GetSignedPubKeysFromBitmap(self, bitmap: bytes):
        if self.Len() != len(bitmap):
            raise ValueError(f"mismatching bitmap lengths expectedBitmapLength {self.Len()} providedBitmapLength {len(bitmap)}")
        return [p for i, p in enumerate(self.Publics) if bitmap[i >> 3] & (1 << (i & 7))]
    def IndexEnabled(self, i: int) -> bool:
        if i >= len(self.Publics): raise IndexError("index out of range")
        return (self.Bitmap[i >> 3] & (1 << (i & 7))) != 0
    def KeyEnabled(self, public: bytes) -> bool:
        if public not in self.PublicsIndex: raise KeyError("key not found")
        return self.IndexEnabled(self.PublicsIndex[public])
    def SetKey(self, public: bytes, enable: bool):
        if public not in self.PublicsIndex: raise KeyError("key not found")
        self.SetBit(self.PublicsIndex[public], enable)
    def SetKeysAtomic(self, publics, enable: bool):
        idx = []
        for k in publics:
            if k.Bytes not in self.PublicsIndex: raise KeyError("key not found")
            idx.append(self.PublicsIndex[k.Bytes])
        for i in idx: self.SetBit(i, enable)
    def CountEnabled(self) -> int:
        return sum(1 for i in range(len(self.Publics)) if self.Bitmap[i >> 3] & (1 << (i & 7)))
    def CountTotal(self) -> int: return len(self.Publics)

def NewMask(publics) -> Mask: return Mask(publics)

def AggregateMasks(a: bytes, b: bytes) -> bytes:
    if len(a) != len(b): raise ValueError("mismatching Bitmap lengths")
    return bytes(x | y for x, y in zip(a, b))

class CompletePolicy:
    def Check(self, m: Mask) -> bool: return m.CountEnabled() == m.CountTotal()
class ThresholdPolicy:
    def __init__(self, thold: int): self.thold = thold
    def Check(self, m: Mask) -> bool: return m.CountEnabled() >= self.thold
def NewThresholdPolicy(thold: int): return ThresholdPolicy(thold)

def ConstructCommitPayload(is_staking: bool, block_hash: bytes, block_num: int, view_id: int) -> bytes:
    """consensus/signature/signature.go:12-24."""
    out = block_num.to_bytes(8, "little") + bytes(block_hash)
    if is_staking: out += view_id.to_bytes(8, "little")
    return out

def SelfTestSplit(iters: int = 16) -> int: return int(_need().hbls_selftest_split(iters))
def SetBatchMode(mode: int): lib().hbls_set_batch_mode(int(mode))
def GetBatchMode() -> int: return int(lib().hbls_get_batch_mode())
def BuildInfo() -> dict:
    v = int(lib().hbls_build_info()); return {"batch_inv": bool(v & 1), "batch_k": v >> 8}
def KernelLaunchCount() -> int: return int(lib().hbls_kernel_launch_count())
def ProbeMac32PerS(iters: int = 4096):
    """(achieved IMAD.WIDE MAC32/s of the carry-chain probe, SM clock in Hz measured under that load)."""
    clk = ctypes.c_double(0.0)
    v = float(_need().hbls_probe_mac32_per_s(iters, ctypes.byref(clk)))
    return v, float(clk.value)
def LastBatchInfo() -> dict:
    bi = BatchInfo()
    rc = lib().hbls_last_batch_info(ctypes.byref(bi))
    if rc != 0: raise HblsError(f"hbls_last_batch_info rc={rc}")
    return bi.as_dict()
def SetParam(name: str, value: int):
    if lib().hbls_set_param(name.encode(), int(value)) != 0: raise ValueError(f"hbls_set_param({name}, {value})")
def GetParam(name: str) -> int: return int(lib().hbls_get_param(name.encode()))
def LastError():
    buf = ctypes.create_string_buffer(160)
    return int(lib().hbls_last_error(buf, 160)), buf.value.decode()

class DeviceMask:
    """Persistent device Mask (hbls_mask_*): crypto/bls/mask.go semantics with the running aggregate key resident in HBM;
    SetMask / SetBit apply only the delta (SURVEY 8f.2, TODO(audit) consensus/consensus_service.go:318)."""
    def __init__(self, committee: Committee):
        self.c = committee; self.h = ctypes.c_void_p()
        rc = _need().hbls_mask_create(ctypes.byref(self.h), committee.h)
        if rc != 0: raise HblsError(f"hbls_mask_create rc={rc}")
    def __del__(self):
        try:
            if self.h and _lib is not None: _lib.hbls_mask_destroy(self.h); self.h = None
        except Exception: pass
    def Len(self): return self.c.blen()
    def SetMask(self, mask: bytes):
        rc = _lib.hbls_mask_set_mask(self.h, _buf(mask), len(mask))
        if rc == ERR_ARG: raise ValueError(f"mismatching bitmap lengths expectedBitmapLength {self.Len()} providedBitmapLength {len(mask)}")
        if rc != 0: raise HblsError(f"hbls_mask_set_mask rc={rc}")
    def SetBit(self, i: int, enable: bool):
        rc = _lib.hbls_mask_set_bit(self.h, i, 1 if enable else 0)
        if rc == ERR_ARG: raise IndexError("index out of range")
        if rc != 0: raise HblsError(f"hbls_mask_set_bit rc={rc}")
    def Clear(self):
        if _lib.hbls_mask_clear(self.h) != 0: raise HblsError("hbls_mask_clear")
    def CountEnabled(self) -> int: return int(_lib.hbls_mask_count_enabled(self.h))
    def Mask(self) -> bytes:
        out = ctypes.create_string_buffer(self.Len() if self.Len() else 1)
        if _lib.hbls_mask_get(self.h, out, self.Len(), None) != 0: raise HblsError("hbls_mask_get")
        return out.raw[:self.Len()]
    def AggregatePublicBytes(self) -> bytes:
        out = ctypes.create_string_buffer(48)
        if _lib.hbls_mask_get(self.h, None, 0, out) != 0: raise HblsError("hbls_mask_get")
        return out.raw
    def VerifyHash(self, sig96: bytes, msg: bytes) -> bool:
        rc = _lib.hbls_mask_verify(self.h, _buf(sig96), _buf(msg), len(msg))
        if rc < 0: raise HblsError(f"hbls_mask_verify rc={rc}")
        return rc == 1

class BallotBox:
    """Running vote aggregate (hbls_ballot_box_*): quorum.go:164-196 AggregateVotes with each vote decoded once on arrival."""
    def __init__(self, committee: Committee):
        self.c = committee; self.h = ctypes.c_void_p()
        rc = _need().hbls_ballot_box_create(ctypes.byref(self.h), committee.h)
        if rc != 0: raise HblsError(f"hbls_ballot_box_create rc={rc}")
    def __del__(self):
        try:
            if self.h and _lib is not None: _lib.hbls_ballot_box_destroy(self.h); self.h = None
        except Exception: pass
    def AddVote(self, signer_bitmap: bytes, sig96: bytes) -> bool:
        """True if counted, False if skipped (a signer was already collected); ValueError on an undecodable signature."""
        rc = _lib.hbls_ballot_box_add_vote(self.h, _buf(signer_bitmap), len(signer_bitmap), _buf(sig96))
        if rc == ERR_DECODE: raise ValueError("err blsSignatureDeserialize")
        if rc < 0: raise HblsError(f"hbls_ballot_box_add_vote rc={rc}")
        return rc == 0
    def Aggregate(self):
        sig = ctypes.create_string_buffer(96); bm = ctypes.create_string_buffer(self.c.blen() if self.c.blen() else 1)
        rc = _lib.hbls_ballot_box_aggregate(self.h, sig, bm, self.c.blen())
        if rc != 0: raise HblsError(f"hbls_ballot_box_aggregate rc={rc}")
        return sig.raw, bm.raw[:self.c.blen()]

STAGE_NAMES = ["k_mask_aggregate", "k_g1_normalize", "k_g2_decode", "k_hash_to_g2", "k_rlc_scale+k_rlc_group_sum", "pairing"]
def StageTimingEnable(on: bool): lib().hbls_stage_timing_enable(1 if on else 0)
def StageTimingGet():
    """six stage times (ms) of the last aggregate-verify pipeline issued with stage timing on"""
    buf = (ctypes.c_float * 8)()
    n = lib().hbls_stage_timing_get(buf, 6)
    return [float(buf[i]) for i in range(n)]
def StageTimingLinesMs():
    """the line kernel's share of stage 5 (ms) when the batched pairing ran as two kernels, else 0"""
    buf = (ctypes.c_float * 8)()
    n = lib().hbls_stage_timing_get(buf, 8)
    return float(buf[6]) if n >= 7 else 0.0
