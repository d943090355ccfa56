"""tools/concurrency_bench.py -- throughput and latency of the per-call API (blsVerifyHash, blsSignHash, blsSignatureDeserialize)
called from T threads at once, the way Harmony's goroutines call it.  Every call ends in a device synchronise, so the wall-clock time
around it is the caller's latency.

    python tools/concurrency_bench.py [--lib path/libhbls.so] [--threads 1,2,8,32,128,512]      one library, JSON lines
    python tools/concurrency_bench.py --compare A.so B.so [--rounds 2]                          A and B alternating, table

Per (threads, op): calls/s, p50 / p99 latency (ms) and, where the library counts it (hbls_coalesce_stats), the mean batch size.
ops: verify_distinct (VerifyHash, a different message per call), verify_same (one message for every call), sign (SignHash,
different messages), sig_des (Sign.Deserialize of valid signatures).  Each library runs in its own process."""
import argparse, ctypes, json, os, subprocess, sys, threading, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from harmony_b200 import workload as wl

class Sec(ctypes.Structure): _fields_ = [("d", ctypes.c_uint64 * 4)]
class Pub(ctypes.Structure): _fields_ = [("d", ctypes.c_uint64 * 18)]
class Sig(ctypes.Structure): _fields_ = [("d", ctypes.c_uint64 * 36)]
OPS = ["verify_distinct", "verify_same", "sign", "sig_des"]
POOL = 128

def load(path):
    L = ctypes.CDLL(path); c = ctypes
    L.blsInit.argtypes = [c.c_int, c.c_int]
    L.blsSecretKeyDeserialize.argtypes = [c.POINTER(Sec), c.c_char_p, c.c_size_t]
    L.blsGetPublicKey.argtypes = [c.POINTER(Pub), c.POINTER(Sec)]
    L.blsSignHash.argtypes = [c.POINTER(Sig), c.POINTER(Sec), c.c_char_p, c.c_size_t]
    L.blsVerifyHash.argtypes = [c.POINTER(Sig), c.POINTER(Pub), c.c_char_p, c.c_size_t]
    L.blsSignatureSerialize.argtypes = [c.c_void_p, c.c_size_t, c.POINTER(Sig)]
    L.blsSignatureDeserialize.argtypes = [c.POINTER(Sig), c.c_char_p, c.c_size_t]
    L.blsSignatureSerialize.restype = L.blsSignatureDeserialize.restype = c.c_size_t
    stats = None
    if hasattr(L, "hbls_coalesce_stats"):
        L.hbls_coalesce_stats.argtypes = [c.POINTER(c.c_uint64)] * 3
        def stats():
            r, b, m = c.c_uint64(), c.c_uint64(), c.c_uint64()
            L.hbls_coalesce_stats(c.byref(r), c.byref(b), c.byref(m)); return r.value, b.value
    return L, stats

def setup(L):
    assert L.blsInit(5, 46) == 0, "blsInit failed"
    secs, pubs = [], []
    for i in range(8):
        s = Sec(); assert L.blsSecretKeyDeserialize(ctypes.byref(s), wl.sk_bytes(wl.seeded_sk("cbench", i)), 32) == 32
        p = Pub(); L.blsGetPublicKey(ctypes.byref(p), ctypes.byref(s)); secs.append(s); pubs.append(p)
    msgs = [wl.seeded_bytes("cbench/m", j, 48) for j in range(POOL)]
    sigs, ser = [], []
    for j in range(POOL):
        s = Sig(); assert L.blsSignHash(ctypes.byref(s), ctypes.byref(secs[j % 8]), msgs[j], 48) == 0
        b = ctypes.create_string_buffer(96); L.blsSignatureSerialize(b, 96, ctypes.byref(s)); sigs.append(s); ser.append(b.raw)
    return secs, pubs, msgs, sigs, ser

def call(L, ctx, op, n):
    secs, pubs, msgs, sigs, ser = ctx
    j = n % POOL
    if op == "verify_distinct": assert L.blsVerifyHash(ctypes.byref(sigs[j]), ctypes.byref(pubs[j % 8]), msgs[j], 48) == 1
    elif op == "verify_same": assert L.blsVerifyHash(ctypes.byref(sigs[0]), ctypes.byref(pubs[0]), msgs[0], 48) == 1
    elif op == "sign": out = Sig(); assert L.blsSignHash(ctypes.byref(out), ctypes.byref(secs[j % 8]), msgs[j], 48) == 0
    else: out = Sig(); assert L.blsSignatureDeserialize(ctypes.byref(out), ser[j], 96) == 96

def measure(L, stats, ctx, op, T, target):
    per = max(2, -(-target // T))
    lat = [[] for _ in range(T)]; bar = threading.Barrier(T + 1); err = []
    def w(t):
        try:
            bar.wait()
            for i in range(per):
                t0 = time.perf_counter(); call(L, ctx, op, t * per + i); lat[t].append(time.perf_counter() - t0)
        except BaseException as e:      # noqa: BLE001
            err.append(e)
    th = [threading.Thread(target=w, args=(t,), daemon=True) for t in range(T)]
    for x in th: x.start()
    s0 = stats() if stats else None
    bar.wait(); t0 = time.perf_counter()
    for x in th: x.join()
    wall = time.perf_counter() - t0
    if err: raise err[0]
    s1 = stats() if stats else None
    all_lat = sorted(x for row in lat for x in row)
    q = lambda f: all_lat[min(len(all_lat) - 1, int(f * len(all_lat)))] * 1e3
    res = {"op": op, "threads": T, "calls": len(all_lat), "calls_per_s": round(len(all_lat) / wall, 1), "p50_ms": round(q(0.5), 3), "p99_ms": round(q(0.99), 3)}
    if s1: res["mean_batch"] = round((s1[0] - s0[0]) / max(1, s1[1] - s0[1]), 2)
    return res

def run_one(path, threads, target):
    L, stats = load(path)
    ctx = setup(L)
    for op in OPS:                                     # warm-up: first launches, scratch growth, H(m) cache
        for i in range(8): call(L, ctx, op, i)
        measure(L, stats, ctx, op, 8, 16)
    for T in threads:
        for op in OPS:
            print(json.dumps({"lib": os.path.basename(path), **measure(L, stats, ctx, op, T, target)}), flush=True)

def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        return out.strip().splitlines()[0]
    except Exception:                                  # noqa: BLE001
        return "unknown"

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=os.path.join(ROOT, "harmony_b200", "lib", "libhbls.so"))
    ap.add_argument("--threads", default="1,2,8,32,128,512")
    ap.add_argument("--target", type=int, default=256, help="calls per (threads, op), at least 2 per thread")
    ap.add_argument("--compare", nargs=2, metavar=("A", "B"))
    ap.add_argument("--rounds", type=int, default=2)
    a = ap.parse_args()
    if not a.compare:
        run_one(a.lib, [int(x) for x in a.threads.split(",")], a.target); return
    print(f"# GPU: {gpu_info()}", flush=True)
    rows = {}
    for r in range(a.rounds):
        for lib in a.compare:                          # alternating, each in a fresh process
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--lib", lib, "--threads", a.threads, "--target", str(a.target)],
                                 stdout=subprocess.PIPE, text=True, check=True).stdout
            for line in out.splitlines():
                d = json.loads(line); rows.setdefault((d["op"], d["threads"], lib), []).append(d)
                print(f"# round {r} {line}", flush=True)
    names = [os.path.basename(os.path.dirname(os.path.abspath(x))) + "/" + os.path.basename(x) for x in a.compare]
    print(f"{'op':16s} {'threads':>7s} | " + " | ".join(f"{n[-28:]:>28s} calls/s (min..max)  p50 ms  p99 ms  batch" for n in names))
    for op in OPS:
        for T in [int(x) for x in a.threads.split(",")]:
            cells = []
            for lib in a.compare:
                rs = rows[(op, T, lib)]
                cps = [x["calls_per_s"] for x in rs]
                med = lambda k: sorted(x[k] for x in rs)[len(rs) // 2]
                cells.append(f"{min(cps):10.1f}..{max(cps):<10.1f} {med('p50_ms'):8.3f} {med('p99_ms'):7.3f} {str(rs[0].get('mean_batch', '-')):>6s}")
            print(f"{op:16s} {T:7d} | " + " | ".join(f"{c:>61s}" for c in cells), flush=True)

if __name__ == "__main__":
    main()
