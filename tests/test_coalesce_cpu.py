"""CPU-only checks of the coalesced per-call operations (include/hbls.h "Threading"):

- the request combiner (harmony_b200/csrc/coalesce.hpp) with a fake executor, built under ThreadSanitizer and AddressSanitizer, from
  64 threads x 5 000 requests: every caller gets its own result, nothing hangs, a lone caller runs batches of one itself, contended
  batches exceed one request but never the cap, and no thread runs a batch that does not hold its own request;
- the device code of the batched passes run on the host (tests/emu/emu_coalesce.cpp): k_hm_gather, and the struct-layout decode
  against the one-thread deserializers, byte for byte, for valid, identity, undecodable and on-curve non-subgroup encodings."""
import ctypes, os, random, subprocess
import pytest
from harmony_b200 import workload as wl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "emu")
P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab

@pytest.mark.parametrize("sanitizer", ["thread", "address"])
def test_combiner_fake_executor(sanitizer, tmp_path):
    exe = str(tmp_path / f"coalesce_fake_{sanitizer}")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-g", f"-fsanitize={sanitizer}", "-pthread", "-o", exe,
                           os.path.join(EMU, "coalesce_fake.cpp")])
    for cap in ("16", "4096"):
        r = subprocess.run([exe, "64", "5000", cap], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "all checks passed" in r.stdout, r.stdout + r.stderr
        assert "WARNING: ThreadSanitizer" not in r.stderr and "ERROR: AddressSanitizer" not in r.stderr, r.stderr

@pytest.fixture(scope="module")
def emuc(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu") / "libhbls_emu_coalesce.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-o", out, os.path.join(EMU, "emu_coalesce.cpp")])
    L = ctypes.CDLL(out)
    L.emu_hm_gather.argtypes = [ctypes.c_size_t, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_size_t, ctypes.c_void_p]
    L.emu_decode_struct_g2.argtypes = [ctypes.c_size_t, ctypes.c_char_p, ctypes.c_void_p]
    L.emu_decode_struct_g1.argtypes = [ctypes.c_size_t, ctypes.c_char_p, ctypes.c_void_p]
    return L

def test_hm_gather_duplicate_and_unique_messages(emuc):
    msgs = [wl.commit_payload("hmg", i) for i in range(4)] + [bytes(48)]          # the last maps to no point (ok flag 0)
    idx = [0, 1, 1, 2, 0, 4, 3, 3, 3, 1, 4, 2]
    arr = (ctypes.c_uint32 * len(idx))(*idx)
    assert emuc.emu_hm_gather(len(msgs), b"".join(msgs), 48, len(idx), arr) == 1
    one = (ctypes.c_uint32 * 1)(2)
    assert emuc.emu_hm_gather(len(msgs), b"".join(msgs), 48, 1, one) == 1

def _on_curve_g1(rng):
    """48-byte encoding of a point on y^2 = x^3 + 4 that is (with overwhelming probability) outside the order-r subgroup."""
    while True:
        x = rng.randrange(1, P)
        if pow((x ** 3 + 4) % P, (P - 1) // 2, P) == 1:
            b = bytearray(x.to_bytes(48, "little")); b[47] |= rng.choice([0, 0x80]); return bytes(b)

def _fp2_mul(a, b):
    return ((a[0] * b[0] - a[1] * b[1]) % P, (a[0] * b[1] + a[1] * b[0]) % P)

def _on_curve_g2(rng):
    """96-byte encoding of a point on y^2 = x^3 + 4(1 + i) outside the subgroup: x^3 + b is a square in Fp2 iff its norm is one in Fp."""
    while True:
        x = (rng.randrange(P), rng.randrange(1, P))
        t = _fp2_mul(_fp2_mul(x, x), x); t = ((t[0] + 4) % P, (t[1] + 4) % P)
        if pow((t[0] * t[0] + t[1] * t[1]) % P, (P - 1) // 2, P) == 1:
            b = bytearray(x[0].to_bytes(48, "little") + x[1].to_bytes(48, "little")); b[95] |= rng.choice([0, 0x80]); return bytes(b)

def test_signature_struct_decode_matches_one_thread_deserialize(emuc, oracle):
    rng = random.Random(11)
    sks = [wl.sk_bytes(wl.seeded_sk("des2", i)) for i in range(3)]
    sigs = [oracle.sign_hash(s, wl.commit_payload("des2", i)) for i, s in enumerate(sks)]
    sigs += [bytes(96), b"\xff" * 96, _on_curve_g2(rng), _on_curve_g2(rng), rng.randbytes(96)]
    cls = ctypes.create_string_buffer(len(sigs))
    assert emuc.emu_decode_struct_g2(len(sigs), b"".join(sigs), cls) == len(sigs)
    got = list(cls.raw)
    assert got[:4] == [1, 1, 1, 1] and got[4] == 3 and got[5:7] == [2, 2], got

def test_public_key_struct_decode_matches_one_thread_deserialize(emuc, oracle):
    rng = random.Random(12)
    pks = [oracle.get_public_key(wl.sk_bytes(wl.seeded_sk("des1", i))) for i in range(3)]
    pks += [bytes(48), b"\xff" * 48, _on_curve_g1(rng), _on_curve_g1(rng), rng.randbytes(48)]
    cls = ctypes.create_string_buffer(len(pks))
    assert emuc.emu_decode_struct_g1(len(pks), b"".join(pks), cls) == len(pks)
    got = list(cls.raw)
    assert got[:4] == [1, 1, 1, 1] and got[4] == 3 and got[5:7] == [2, 2], got
