// harmony_b200/csrc/kernels.cuh -- __global__ entry points of the BLS hot path (thread-per-item throughput kernels).
//
// Data layout in HBM (all arrays of structs, Montgomery limbs, little-endian u32):
//   g1a  96 B  affine G1   (committee table rows, -apk per round)
//   g2a 192 B  affine G2   (decoded signatures, H(m))
//   g1  144 B / g2 288 B   Jacobian partial sums
//   fp12 576 B             Miller-loop outputs, 2 per verification round
// The arithmetic is integer-pipe bound (~375 MAC32 per byte touched, SURVEY 8d): HBM is idle by design; the
// launch geometry therefore only aims at filling 148 SMs x 4 schedulers with independent IMAD chains.
#pragma once
#include "pairing.cuh"
#include "vm.cuh"

namespace hb {

#ifndef HB_MINBLOCKS
#define HB_MINBLOCKS 4      // 64-thread CTAs: 4 => up to 255 regs/thread, 8 => 128
#endif
#define HB_TID ((size_t)blockIdx.x * blockDim.x + threadIdx.x)
#define HB_STRIDE ((size_t)gridDim.x * blockDim.x)      // heavy kernels are persistent grid-stride loops: resident threads are capped
                                                        // so the per-thread working set (~3 KB of Fp12 temporaries) stays in L1/L2

// ---- parity probe: canonical LE operands -> Montgomery -> product -> canonical
__global__ void k_fp_mul(size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out) {
    size_t i = HB_TID; if (i >= n) return;
    fp x, y, v;
    load_words(v.l, a + 48 * i, 12); fp_from_int(x, v);
    load_words(v.l, b + 48 * i, 12); fp_from_int(y, v);
    fp_mul(x, x, y); fp_to_int(v, x); store_words(out + 48 * i, v.l, 12);
}

// ---- decode (R2/R3 of SURVEY 8a): 48/96 B -> affine point (+ optional negation), ok flag
__global__ void k_g1_decode(size_t n, const uint8_t* in, g1a* out, uint8_t* ok, int check_order, int negate) {
    size_t i = HB_TID; if (i >= n) return;
    g1 p; bool good = g1_deserialize(p, in + 48 * i, check_order != 0);
    g1a a;
    if (!good || pt_is_inf(p)) { fp_zero(a.x); fp_zero(a.y); }
    else { a.x = p.x; a.y = p.y; if (negate) fp_neg(a.y, a.y); }      // deserialize returns z == 1
    out[i] = a; ok[i] = good ? 1 : 0;
}
// triples (hbls_verify_batch): the key feeds the same pipeline as a mask aggregate, so it is kept Jacobian (z = 1; identity on failure)
__global__ void k_g1_decode_jac(size_t n, const uint8_t* in, g1* out, uint8_t* ok, int check_order) {
  for (size_t i = HB_TID; i < n; i += HB_STRIDE) {
    g1 p; bool good = g1_deserialize(p, in + 48 * i, check_order != 0);
    if (!good) pt_set_inf(p);
    out[i] = p; ok[i] = good ? 1 : 0;
  }
}
#ifndef HB_DEC_MINBLOCKS
#define HB_DEC_MINBLOCKS 8          // <= 128 registers: 512 resident threads per SM = exactly 4 waves of the 303 104-round batch (30.97 -> 30.30 ms)
#endif
__global__ void __launch_bounds__(64, HB_DEC_MINBLOCKS) k_g2_decode(size_t n, const uint8_t* in, g2a* out, uint8_t* ok, int check_order) {
  for (size_t i = HB_TID; i < n; i += HB_STRIDE) {
    g2 p; bool good = g2_deserialize(p, in + 96 * i, check_order != 0);
    g2a a;
    if (!good || pt_is_inf(p)) { fp2_zero(a.x); fp2_zero(a.y); }
    else { a.x = p.x; a.y = p.y; }
    out[i] = a; ok[i] = good ? 1 : 0;
  }
}

// subgroup test of already-decoded affine points, one per thread (second half of k_g2_decode when the stage runs as two kernels,
// hbls.cu "decode_split": square-root chains | G2 ladder); a point outside the subgroup loses its ok flag and is zeroed
__global__ void __launch_bounds__(64, HB_DEC_MINBLOCKS) k_g2_subgroup(size_t n, g2a* pts, uint8_t* ok) {
  for (size_t i = HB_TID; i < n; i += HB_STRIDE) {
    if (!ok[i]) continue;
    const g2a a = pts[i];
    if (aff_is_inf(a)) continue;
    g2 q; q.x = a.x; q.y = a.y; fp2_one(q.z);
    if (!g2_in_subgroup(q)) { g2a z; fp2_zero(z.x); fp2_zero(z.y); pts[i] = z; ok[i] = 0; }
  }
}

// ---- warp shuffle of a whole point
template <class T> HB_DEV void shfl_down_struct(T& dst, const T& src, int off) {
    const uint32_t* s = reinterpret_cast<const uint32_t*>(&src);
    uint32_t* d = reinterpret_cast<uint32_t*>(&dst);
    for (int w = 0; w < (int)(sizeof(T) / 4); w++) d[w] = __shfl_down_sync(0xffffffffu, s[w], off);
}

// ---- Mask.SetMask (R4): one warp per round; lane l sums table rows l, l+32, ... whose bit is set, then a
// 5-level shuffle tree folds the 32 partial sums.  Summation order is free: only Serialize normalises (A.6).
__global__ void k_mask_aggregate(size_t B, size_t n, const g1a* __restrict__ table, const uint8_t* __restrict__ bitmaps, size_t blen, g1* out) {
    size_t warp = HB_TID >> 5; int lane = threadIdx.x & 31;
    if (warp >= B) return;
    const uint8_t* bm = bitmaps + warp * blen;
    g1 acc; pt_set_inf(acc);
    for (size_t i = lane; i < n; i += 32) {
        if (bm[i >> 3] & (1u << (i & 7))) { g1a q = table[i]; pt_add_mixed(acc, acc, q); }
    }
    for (int off = 16; off >= 1; off >>= 1) {
        g1 other; shfl_down_struct(other, acc, off);
        if (lane < off) pt_add(acc, acc, other);
    }
    if (lane == 0) out[warp] = acc;
}
// multi-committee form (crosslinks / multi-shard block seal: internal/chain/engine.go:592-604, node/harmony/node_cross_link.go:69-90):
// every item names its own committee table; one warp per item
struct mask_item { const g1a* table; const uint8_t* bitmap; uint64_t n; };
__global__ void k_mask_aggregate_items(size_t B, const mask_item* __restrict__ items, g1* out) {
    size_t warp = HB_TID >> 5; int lane = threadIdx.x & 31;
    if (warp >= B) return;
    const mask_item it = items[warp];
    g1 acc; pt_set_inf(acc);
    for (size_t i = lane; i < it.n; i += 32) {
        if (it.bitmap[i >> 3] & (1u << (i & 7))) { g1a q = it.table[i]; pt_add_mixed(acc, acc, q); }
    }
    for (int off = 16; off >= 1; off >>= 1) {
        g1 other; shfl_down_struct(other, acc, off);
        if (lane < off) pt_add(acc, acc, other);
    }
    if (lane == 0) out[warp] = acc;
}
// large-batch form: one thread per round.  Quorum bitmaps are dense (167..250 of 250 set), so the thread sums whichever
// side is SMALLER -- the set bits, or the unset bits subtracted from the committee total (computed once at
// hbls_committee_create) -- from a compacted index list: ~44 point additions per round instead of ~206, and the
// loop trip counts of the 32 lanes are short and similar.  Group arithmetic only; Serialize normalises (SURVEY A.6).
#define HB_MASK_LIST 512
// The 32 lanes of a warp run as long as the lane with the most additions (167 / 200 / 250 signers of 250 = 83 / 50 / 0 additions:
// ncu showed the multiplier 82 % busy for work worth 43 %).  `order` (nullable) = the rounds sorted by the number of additions they
// need (counting sort on the device: k_mask_count -> k_mask_scan -> k_mask_scatter), so that neighbouring lanes get equal trip counts.
#define HB_MASK_BINS 1024
__global__ void k_mask_count(size_t B, size_t n, const uint8_t* __restrict__ bitmaps, size_t blen, uint16_t* cost, unsigned* hist) {
    const size_t j = HB_TID; if (j >= B) return;
    const uint8_t* bm = bitmaps + j * blen;
    uint32_t k = 0;
    for (size_t i = 0; i < n; i++) k += (bm[i >> 3] >> (i & 7)) & 1u;
    uint32_t c = (2 * (size_t)k > n) ? (uint32_t)(n - k) : k;            // the side k_mask_aggregate_serial will sum
    if (c >= HB_MASK_BINS) c = HB_MASK_BINS - 1;
    cost[j] = (uint16_t)c; atomicAdd(&hist[c], 1u);
}
__global__ void k_mask_scan(unsigned* hist) {                             // exclusive prefix sum of the bins, one thread (1 024 adds)
    if (HB_TID != 0) return;
    unsigned acc = 0;
    for (int i = 0; i < HB_MASK_BINS; i++) { const unsigned h = hist[i]; hist[i] = acc; acc += h; }
}
__global__ void k_mask_scatter(size_t B, const uint16_t* cost, unsigned* hist, uint32_t* order) {
    const size_t j = HB_TID; if (j >= B) return;
    order[atomicAdd(&hist[cost[j]], 1u)] = (uint32_t)j;
}
__global__ void k_mask_aggregate_serial(size_t B, size_t n, const g1a* __restrict__ table, const g1* __restrict__ total,
                                        const uint8_t* __restrict__ bitmaps, size_t blen, g1* out, const uint32_t* __restrict__ order = nullptr) {
  for (size_t jt = HB_TID; jt < B; jt += HB_STRIDE) {
    const size_t j = order ? order[jt] : jt;
    const uint8_t* bm = bitmaps + j * blen;
    uint32_t k = 0;
    for (size_t i = 0; i < n; i++) k += (bm[i >> 3] >> (i & 7)) & 1u;
    const bool fits = n <= 65536;                                                             // idx[] holds 16-bit row numbers
    const bool comp = fits && (2 * (size_t)k > n) && (n - k) <= HB_MASK_LIST && total != nullptr;     // sum the unset side
    g1 acc; pt_set_inf(acc);
    if (comp || (fits && k <= HB_MASK_LIST)) {
        uint16_t idx[HB_MASK_LIST]; uint32_t cnt = 0;
        const uint32_t want = comp ? 0u : 1u;
        for (size_t i = 0; i < n; i++) if (((bm[i >> 3] >> (i & 7)) & 1u) == want) idx[cnt++] = (uint16_t)i;
        for (uint32_t t = 0; t < cnt; t++) { g1a q = table[idx[t]]; pt_add_mixed(acc, acc, q); }
        if (comp) { g1 tot = *total; pt_neg(acc, acc); pt_add(acc, tot, acc); }
    } else {
        for (size_t i = 0; i < n; i++) if ((bm[i >> 3] >> (i & 7)) & 1u) { g1a q = table[i]; pt_add_mixed(acc, acc, q); }
    }
    out[j] = acc;
  }
}
// committee total (sum of all table rows), single CTA
__global__ void __launch_bounds__(128) k_g1_sum(size_t n, const g1a* in, g1* out) {
    __shared__ g1 sm[128];
    g1 acc; pt_set_inf(acc);
    for (size_t i = threadIdx.x; i < n; i += 128) { g1a q = in[i]; pt_add_mixed(acc, acc, q); }
    sm[threadIdx.x] = acc;
    __syncthreads();
    for (int off = 64; off >= 1; off >>= 1) {
        if ((int)threadIdx.x < off) { g1 o = sm[threadIdx.x + off]; pt_add(acc, acc, o); sm[threadIdx.x] = acc; }
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = acc;
}
__global__ void k_g1_normalize(size_t n, const g1* in, g1a* out, int negate, const int* run_if) {
    if (run_if && !*run_if) return;          // deferred form: only needed when the batched check sends rounds to the exact pass
    size_t i = HB_TID; if (i >= n) return;
    g1 p = in[i]; g1a a; pt_to_aff(a, p);
    if (negate) fp_neg(a.y, a.y);
    out[i] = a;
}
// latency path: affine -apk with the binary-GCD inverse
__global__ void k_g1_normalize_lat(size_t n, const g1* in, g1a* out, int negate) {
    size_t i = HB_TID; if (i >= n) return;
    g1 p = in[i]; g1a a;
    if (pt_is_inf(p)) { fp_zero(a.x); fp_zero(a.y); }
    else {
        fp zi, zi2; fp_inv_gcd(zi, p.z); fp_sqr(zi2, zi);
        fp_mul(a.x, p.x, zi2); fp_mul(zi2, zi2, zi); fp_mul(a.y, p.y, zi2);
        if (negate) fp_neg(a.y, a.y);
    }
    out[i] = a;
}
__global__ void k_g2_normalize(size_t n, const g2* in, g2a* out) {
    size_t i = HB_TID; if (i >= n) return;
    g2 p = in[i]; g2a a; pt_to_aff(a, p);
    out[i] = a;
}
__global__ void k_g1_serialize(size_t n, const g1* in, uint8_t* out) {
    size_t i = HB_TID; if (i >= n) return;
    g1 p = in[i]; g1_serialize(out + 48 * i, p);
}
__global__ void k_g2_serialize(size_t n, const g2* in, uint8_t* out) {
    size_t i = HB_TID; if (i >= n) return;
    g2 p = in[i]; g2_serialize(out + 96 * i, p);
}

// ---- AggregateSig (R5): single-CTA strided sum + shared-memory tree; out = 1 Jacobian point
#define HB_SUM_THREADS 128
__global__ void __launch_bounds__(HB_SUM_THREADS) k_g2_sum(size_t n, const g2a* in, g2* out) {
    __shared__ g2 sm[HB_SUM_THREADS];
    g2 acc; pt_set_inf(acc);
    for (size_t i = threadIdx.x; i < n; i += HB_SUM_THREADS) { g2a q = in[i]; pt_add_mixed(acc, acc, q); }
    sm[threadIdx.x] = acc;
    __syncthreads();
    for (int off = HB_SUM_THREADS / 2; off >= 1; off >>= 1) {
        if ((int)threadIdx.x < off) { g2 o = sm[threadIdx.x + off]; pt_add(acc, acc, o); sm[threadIdx.x] = acc; }
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = acc;
}

// ---- message -> G2 (hash part of R6/R7), affine output
// HB_BATCH_INV: a persistent thread shares ONE inversion among HB_BATCH_K of its items (Montgomery's trick) -- both inversions of
// hash-to-G2 and the affine conversion of the coefficient-scaling stage.  Measured on B200 at 303 104 rounds/step (profiles/
// r2_stage_times.txt): off 251.3 ms, K = 4 248.2 ms, K = 8 243.2 ms per step.
#ifndef HB_BATCH_INV
#define HB_BATCH_INV 1
#endif
#ifndef HB_BATCH_K
#define HB_BATCH_K 8
#endif
__global__ void k_hash_to_g2(size_t n, const uint8_t* msgs, uint32_t msg_len, g2a* out, uint8_t* ok) {
#if HB_BATCH_INV
  for (size_t i0 = HB_TID; i0 < n; i0 += (size_t)HB_BATCH_K * HB_STRIDE) {
    g2 h[HB_BATCH_K]; fp2 z[HB_BATCH_K], t[HB_BATCH_K], u[HB_BATCH_K], ct[HB_BATCH_K]; bool skip[HB_BATCH_K], good[HB_BATCH_K];
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t i = i0 + (size_t)k * HB_STRIDE;
        good[k] = false; skip[k] = true;
        if (i >= n) continue;
        fp_zero(t[k].b); hash_to_fp(t[k].a, msgs + (size_t)msg_len * i, msg_len);
        good[k] = sw_map_g2_pre(u[k], ct[k], z[k], t[k]);
        skip[k] = !good[k];
    }
    f_batch_inv<fp2, HB_BATCH_K>(z, skip);                     // the maps' (u c1 t)^-1
    for (int k = 0; k < HB_BATCH_K; k++) {
        if (skip[k]) continue;
        g2 a;
        good[k] = sw_map_g2_post(a, t[k], u[k], ct[k], z[k]);
        if (good[k]) g2_clear_cofactor(h[k], a);
        skip[k] = !good[k] || pt_is_inf(h[k]);
        if (!skip[k]) z[k] = h[k].z;
    }
    f_batch_inv<fp2, HB_BATCH_K>(z, skip);                     // -> affine
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t i = i0 + (size_t)k * HB_STRIDE;
        if (i >= n) continue;
        g2a a;
        if (skip[k]) { fp2_zero(a.x); fp2_zero(a.y); } else pt_to_aff_zinv(a, h[k], z[k]);
        out[i] = a; ok[i] = good[k] ? 1 : 0;
    }
  }
#else
  for (size_t i = HB_TID; i < n; i += HB_STRIDE) {
    g2 h; bool good = map_to_g2(h, msgs + (size_t)msg_len * i, msg_len);
    g2a a;
    if (!good) { fp2_zero(a.x); fp2_zero(a.y); } else pt_to_aff(a, h);
    out[i] = a; ok[i] = good ? 1 : 0;
  }
#endif
}

// ---- the same hash in two kernels (large batches, hbls.cu "hash_split"): the Shallue-van de Woestijne map is Fp-only work (square-
// root exponentiation chains, Jacobi symbols, the shared inversion) with a small register and instruction-cache footprint, the
// cofactor clearing is G2 ladders over Fp2.  Separate kernels let the first run with more resident warps and keep each kernel's hot
// code small (ncu on the fused kernel: stall_no_instruction 0.78 per issue, 3 warps per scheduler).
#ifndef HB_SW_MINBLOCKS
#define HB_SW_MINBLOCKS 8         // x 64 threads = 512 resident threads per SM (<= 128 registers); measured 64.6 -> 62.4 ms per 303 104 messages
#endif
__global__ void __launch_bounds__(64, HB_SW_MINBLOCKS) k_hash_sw(size_t n, const uint8_t* msgs, uint32_t msg_len, g2a* pts, uint8_t* ok) {
  for (size_t i0 = HB_TID; i0 < n; i0 += (size_t)HB_BATCH_K * HB_STRIDE) {
    fp2 z[HB_BATCH_K], t[HB_BATCH_K], u[HB_BATCH_K], ct[HB_BATCH_K]; bool skip[HB_BATCH_K];
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t i = i0 + (size_t)k * HB_STRIDE;
        skip[k] = true;
        if (i >= n) continue;
        fp_zero(t[k].b); hash_to_fp(t[k].a, msgs + (size_t)msg_len * i, msg_len);
        skip[k] = !sw_map_g2_pre(u[k], ct[k], z[k], t[k]);
    }
    f_batch_inv<fp2, HB_BATCH_K>(z, skip);
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t i = i0 + (size_t)k * HB_STRIDE;
        if (i >= n) continue;
        g2 a; g2a o; fp2_zero(o.x); fp2_zero(o.y);
        const bool good = !skip[k] && sw_map_g2_post(a, t[k], u[k], ct[k], z[k]);
        if (good) { o.x = a.x; o.y = a.y; }
        pts[i] = o; ok[i] = good ? 1 : 0;
    }
  }
}
// cofactor clearing alone, Jacobian result (no per-thread arrays of pending items: the frame is the group law's own temporaries), and
// the shared-inversion affine conversion as its own small kernel
__global__ void k_hash_cofactor_jac(size_t n, const g2a* pts, const uint8_t* ok, g2* out) {
  for (size_t i = HB_TID; i < n; i += HB_STRIDE) {
    g2 h; pt_set_inf(h);
    if (ok[i]) { g2 a; const g2a p = pts[i]; a.x = p.x; a.y = p.y; fp2_one(a.z); g2_clear_cofactor(h, a); }
    out[i] = h;
  }
}
__global__ void k_g2_normalize_batch(size_t n, const g2* in, g2a* out) {
  for (size_t i0 = HB_TID; i0 < n; i0 += (size_t)HB_BATCH_K * HB_STRIDE) {
    fp2 z[HB_BATCH_K]; bool skip[HB_BATCH_K];
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t i = i0 + (size_t)k * HB_STRIDE;
        skip[k] = true;
        if (i >= n) continue;
        z[k] = in[i].z; skip[k] = fp2_is_zero(z[k]);
    }
    f_batch_inv<fp2, HB_BATCH_K>(z, skip);
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t i = i0 + (size_t)k * HB_STRIDE;
        if (i >= n) continue;
        g2a a;
        if (skip[k]) { fp2_zero(a.x); fp2_zero(a.y); } else { const g2 h = in[i]; pt_to_aff_zinv(a, h, z[k]); }
        out[i] = a;
    }
  }
}
__global__ void k_hash_cofactor(size_t n, g2a* pts, const uint8_t* ok) {
  for (size_t i0 = HB_TID; i0 < n; i0 += (size_t)HB_BATCH_K * HB_STRIDE) {
    g2 h[HB_BATCH_K]; fp2 z[HB_BATCH_K]; bool skip[HB_BATCH_K];
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t i = i0 + (size_t)k * HB_STRIDE;
        skip[k] = true;
        if (i >= n || !ok[i]) continue;
        g2 a; const g2a p = pts[i]; a.x = p.x; a.y = p.y; fp2_one(a.z);
        g2_clear_cofactor(h[k], a);
        skip[k] = pt_is_inf(h[k]);
        if (!skip[k]) z[k] = h[k].z;
    }
    f_batch_inv<fp2, HB_BATCH_K>(z, skip);
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t i = i0 + (size_t)k * HB_STRIDE;
        if (i >= n) continue;
        g2a a;
        if (skip[k]) { fp2_zero(a.x); fp2_zero(a.y); } else pt_to_aff_zinv(a, h[k], z[k]);
        pts[i] = a;
    }
  }
}

// ---- lane-pair forms of decode / hash for small batches (latency path, hbls.cu: B <= coop_max): one item per LANE PAIR.  The Fp-only
// chains (square roots, Jacobi symbols, the SW map) run redundantly on both lanes; the long G2 ladders -- subgroup test, cofactor
// clearing -- run on the split carrier (an Fp2 product costs one product-time per lane instead of three), inversions by binary GCD.
// out_jac (nullable): the decoded point is ALSO written in the blsSignature layout -- the Jacobian struct g2_deserialize returns
// (z = Montgomery one; all zero for the identity) -- for the items that decode; undecodable items leave their struct untouched
// (blsSignatureDeserialize, hbls.cu).  out may then be null.
__global__ void k_g2_decode_pair(size_t n, const uint8_t* in, g2a* out, uint8_t* ok, int check_order, g2* out_jac = nullptr) {
    const size_t i = HB_TID >> 1; if (i >= n) return;                    // a pair leaves together
    g2 p; bool good = g2_deserialize(p, in + 96 * i, false);
    if (good && check_order && !pt_is_inf(p)) {
        jac<fp2h> q; fp2h_pack(q.x, p.x); fp2h_pack(q.y, p.y); fp2h_pack(q.z, p.z);
        good = g2_in_subgroup(q);
    }
    if ((threadIdx.x & 1) == 0) {
        if (out) {
            g2a a;
            if (!good || pt_is_inf(p)) { fp2_zero(a.x); fp2_zero(a.y); } else { a.x = p.x; a.y = p.y; }
            out[i] = a;
        }
        if (out_jac && good) out_jac[i] = p;
        ok[i] = good ? 1 : 0;
    }
}
// per-item H(m) of a coalesced batch (hbls.cu): item i takes the point of its distinct message idx[i]; the host hashed each distinct
// message once (or found it in the H(m) cache)
__global__ void k_hm_gather(size_t n, const uint32_t* idx, const g2a* dist_hm, const uint8_t* dist_ok, g2a* hm, uint8_t* ok) {
    const size_t i = HB_TID; if (i >= n) return;
    const uint32_t d = idx[i];
    hm[i] = dist_hm[d]; ok[i] = dist_ok[d];
}
__global__ void k_hash_to_g2_pair(size_t n, const uint8_t* msgs, uint32_t msg_len, g2a* out, uint8_t* ok) {
    const size_t i = HB_TID >> 1; if (i >= n) return;
    fp2 t; hash_to_fp(t.a, msgs + (size_t)msg_len * i, msg_len); fp_zero(t.b);
    g2 a; bool good = sw_map_g2<true>(a, t);                              // Fp-heavy: both lanes compute the same point
    g2a res; fp2_zero(res.x); fp2_zero(res.y);
    if (good) {
        jac<fp2h> A, H; fp2h_pack(A.x, a.x); fp2h_pack(A.y, a.y); fp2h_pack(A.z, a.z);
        g2_clear_cofactor(H, A);
        if (!pt_is_inf(H)) {
            fp2h zi, zi2, hx, hy; fp2_inv_gcd(zi, H.z); fp2_sqr(zi2, zi);
            fp2_mul(hx, H.x, zi2); fp2_mul(zi2, zi2, zi); fp2_mul(hy, H.y, zi2);
            fp2h_unpack(res.x, hx); fp2h_unpack(res.y, hy);
        }
    }
    if ((threadIdx.x & 1) == 0) { out[i] = res; ok[i] = good ? 1 : 0; }
}
// ---- latency form of hash-to-G2 (vm.cuh): ONE WARP per message.  The Shallue-van de Woestijne map (Fp chains: one inversion, two
// Legendre symbols, the Fp2 square root) runs on every lane alike; the cofactor clearing -- two 63-doubling chains of G2, 52 % of a
// lane pair's hash time (profiles/r2_lat_probe.txt) -- runs as VM step programs with the 3 independent products of a doubling level
// side by side.  Falls back to the complete lane-pair code when the generic formulas degenerate.
__global__ void __launch_bounds__(32) k_hash_to_g2_coop(size_t n, const uint8_t* msgs, uint32_t msg_len, g2a* out, uint8_t* ok, int force_fallback) {
    __shared__ uint32_t slots[VM_SMEM_WORDS];
    const int lane = threadIdx.x & 31;
    vm_load_consts(slots);
    for (size_t i = blockIdx.x; i < n; i += gridDim.x) {
        fp2 t; hash_to_fp(t.a, msgs + (size_t)msg_len * i, msg_len); fp_zero(t.b);
        g2 a; const bool good = sw_map_g2<true>(a, t);                       // warp-uniform: every lane maps the same message
        g2a res; fp2_zero(res.x); fp2_zero(res.y);
        if (good) {
            if (lane == 0) { vm_set_fp2(slots, VM_R_Q2X, a.x); vm_set_fp2(slots, VM_R_Q2Y, a.y); }
            __syncwarp();
            if (vm_hash_cofactor(slots) && !force_fallback) {             // force_fallback: test hook (hbls_set_param "hash_fallback")
                if (lane == 0) { vm_ld(res.x.a.l, slots, VM_R_HX, 0); vm_ld(res.x.b.l, slots, VM_R_HX, 1); vm_ld(res.y.a.l, slots, VM_R_HY, 0); vm_ld(res.y.b.l, slots, VM_R_HY, 1); }
            } else if (lane < 2) {
                jac<fp2h> A, H; fp2h_pack(A.x, a.x); fp2h_pack(A.y, a.y); fp2h_pack(A.z, a.z);
                g2_clear_cofactor(H, A);
                if (!pt_is_inf(H)) {
                    fp2h zi, zi2, hx, hy; fp2_inv_gcd(zi, H.z); fp2_sqr(zi2, zi);
                    fp2_mul(hx, H.x, zi2); fp2_mul(zi2, zi2, zi); fp2_mul(hy, H.y, zi2);
                    fp2h_unpack(res.x, hx); fp2h_unpack(res.y, hy);
                }
            }
        }
        if (lane == 0) { out[i] = res; ok[i] = good ? 1 : 0; }
        __syncwarp();
    }
}

// same-message batches (the leader's prepare / commit vote collection, consensus/leader.go:127-290: every vote signs
// the same block hash / commit payload): H(m) is computed once and replicated
__global__ void k_broadcast_hm(size_t n, g2a* hm, uint8_t* ok) {
    size_t i = HB_TID; if (i == 0 || i >= n) return;
    hm[i] = hm[0]; ok[i] = ok[0];
}

// ---- verification (R7/R8)
// ---- lane-pair form: lanes (2k, 2k+1) co-own round j (even lane = real parts, odd lane = imaginary parts of every Fp2).
// Half the per-thread state of a thread-per-round pairing => twice the warps for the same L1/L2 footprint.  Control flow is
// data-oblivious; rounds with an identity operand (never the case for honest input) are flagged 0xFF and recomputed by
// k_pairing_fixup with the thread-per-round code.
#ifndef HB_TPB_SPLIT
#define HB_TPB_SPLIT 512
#endif
#ifndef HB_MINBLOCKS_SPLIT
#define HB_MINBLOCKS_SPLIT 1        // 1 x 512 threads x 128 regs per SM, lock-stepped per Miller / exponentiation iteration
#endif
__global__ void __launch_bounds__(HB_TPB_SPLIT, HB_MINBLOCKS_SPLIT) k_pairing_verify_split(size_t B, const g2a* sig, const g1a* pk_neg, const g2a* hm,
                                 const uint8_t* ok_a, const uint8_t* ok_b, const uint8_t* ok_c, uint8_t* results, const int* run_if) {
    if (run_if && *run_if == 0) return;                                 // fallback pass of the batched form: nothing failed
    const int role = threadIdx.x & 1;
    const size_t ppg = HB_STRIDE >> 1;                                  // pairs per grid sweep
    for (size_t it = 0; ; it++) {
        const size_t warp_first = it * ppg + ((HB_TID & ~(size_t)31) >> 1);
        if (warp_first >= B) break;                                     // warp-uniform exit
        const size_t j = it * ppg + (HB_TID >> 1);
        const bool valid = j < B;
        const size_t jj = valid ? j : B - 1;
        bool good = (!ok_a || ok_a[jj]) && (!ok_b || ok_b[jj]) && (!ok_c || ok_c[jj]);
        g1a gen, p2 = pk_neg[jj];
        fp_set(gen.x, K_G1_X); fp_set(gen.y, K_G1_Y);
        const fp* s4 = reinterpret_cast<const fp*>(&sig[jj]);           // x.a, x.b, y.a, y.b
        const fp* h4 = reinterpret_cast<const fp*>(&hm[jj]);
        fp2h q1x, q1y, q2x, q2y;
        q1x.c = s4[role]; q1y.c = s4[2 + role]; q2x.c = h4[role]; q2y.c = h4[2 + role];
        // NB: no short-circuit around fp2_is_zero(fp2h) -- it shuffles across the whole warp
        const bool z1x = fp2_is_zero(q1x), z1y = fp2_is_zero(q1y), z2x = fp2_is_zero(q2x), z2y = fp2_is_zero(q2y);
        const bool irregular = (z1x & z1y) | (z2x & z2y) | (fp_is_zero(p2.x) & fp_is_zero(p2.y));
        fp12_t<fp2h> m;
        miller_loop2<fp2h>(m, gen, q1x, q1y, p2, q2x, q2y, true, true);
        final_exp(m, m);
        const bool one = fp12_is_one(m);
        if (valid && role == 0) results[j] = irregular ? 0xFF : ((good && one) ? 1 : 0);
    }
}
// rounds with an identity operand (thread-per-round code path).  An identity public key never verifies (include/hbls.h: a
// zero key would make the zero signature "valid" for every message); an identity signature is checked like any other point.
HB_NOINLINE bool verify_irregular(const g1a& gen, const g2a& q1, const g1a& p2, const g2a& q2) {
    if (aff_is_inf(p2)) return false;
    fp12 m; miller_loop2(m, gen, q1, p2, q2); final_exp(m, m);
    return fp12_is_one(m);
}
__global__ void k_pairing_fixup(size_t B, const g2a* sig, const g1a* pk_neg, const g2a* hm,
                                const uint8_t* ok_a, const uint8_t* ok_b, const uint8_t* ok_c, uint8_t* results, const int* run_if) {
  if (run_if && *run_if == 0) return;
  for (size_t j = HB_TID; j < B; j += HB_STRIDE) {
    if (results[j] != 0xFF) continue;
    bool good = (!ok_a || ok_a[j]) && (!ok_b || ok_b[j]) && (!ok_c || ok_c[j]);
    g1a gen, p2 = pk_neg[j]; g2a q1 = sig[j], q2 = hm[j];
    fp_set(gen.x, K_G1_X); fp_set(gen.y, K_G1_Y);
    results[j] = (good && verify_irregular(gen, q1, p2, q2)) ? 1 : 0;
  }
}
// ---- latency form (vm.cuh): ONE WARP per round runs the 2-pair Miller loop + final exponentiation as step programs over
// shared-memory slots, 16 lane pairs wide.  Same inputs, flags and result protocol as k_pairing_verify_split (0xFF = a round with an
// identity operand, decided afterwards by k_pairing_fixup).  Small batches: a single round is ~10x faster than on one lane pair.
__global__ void __launch_bounds__(32) k_pairing_coop(size_t B, const g2a* sig, const g1a* pk_neg, const g2a* hm,
                                 const uint8_t* ok_a, const uint8_t* ok_b, const uint8_t* ok_c, uint8_t* results) {
    __shared__ uint32_t slots[VM_SMEM_WORDS];
    const int lane = threadIdx.x & 31;
    vm_load_consts(slots);
    for (size_t j = blockIdx.x; j < B; j += gridDim.x) {
        const bool good = (!ok_a || ok_a[j]) && (!ok_b || ok_b[j]) && (!ok_c || ok_c[j]);
        // lanes 0..7 stage one operand each: P1 = generator, Q1 = signature, P2 = -pk, Q2 = H(m)
        bool zero = true;
        if (lane < 8) {
            fp2 v; fp2_zero(v);
            const g1a pk = pk_neg[j];
            switch (lane) {
            case 0: fp_set(v.a, K_G1_X); break;
            case 1: fp_set(v.a, K_G1_Y); break;
            case 2: v = sig[j].x; break;
            case 3: v = sig[j].y; break;
            case 4: v.a = pk.x; break;
            case 5: v.a = pk.y; break;
            case 6: v = hm[j].x; break;
            default: v = hm[j].y; break;
            }
            vm_set_fp2(slots, VM_R_P1X + lane, v);
            zero = fp_is_zero(v.a) & fp_is_zero(v.b);
        }
        const unsigned zmask = __ballot_sync(0xffffffffu, zero);            // bit l: operand l is zero
        const bool irregular = ((zmask & 0x0c) == 0x0c) | ((zmask & 0x30) == 0x30) | ((zmask & 0xc0) == 0xc0);
        bool one = false;
        if (!irregular) one = vm_pairing_check(slots);                        // warp-uniform branch
        if (lane == 0) results[j] = irregular ? 0xFF : ((good && one) ? 1 : 0);
        __syncwarp();
    }
}

// ---- ONE batch split over several GPUs (SURVEY 8e, BASELINE configs[3]): every rank turns its slice into a fixed-size partial record
// { sum_j r_j sigma_j (G2) , prod_j f_{|z|, H_j}(-r_j pk_j) (Fp12, no final exponentiation) , bad count }; the records are all-gathered
// (NCCL) and every rank folds them identically: prod of the partial products x Miller(B, sum of the partial sums), ONE final
// exponentiation.  EC addition / Fp12 multiplication are not NCCL reduction operators, hence all-gather + local fold.
// A warp multiplies the Miller values of its items (w, w + W, ...) into the VM register A; bad / identity items only count.
__global__ void __launch_bounds__(32) k_rlc_partial_coop(size_t n, const g1a* pk_scaled_neg, const g2a* hm, const uint8_t* bad,
                                                         fp2* partial /* 6 per warp, tower order */, unsigned* bad_count) {
    __shared__ uint32_t slots[VM_SMEM_WORDS];
    const int lane = threadIdx.x & 31;
    vm_load_consts(slots);
    vm_run(VM_P_A_ONE, slots);
    for (size_t j = blockIdx.x; j < n; j += gridDim.x) {
        bool zero = true;
        if (lane < 4) {
            fp2 v; fp2_zero(v);
            const g1a pk = pk_scaled_neg[j];
            if (lane == 0) v.a = pk.x; else if (lane == 1) v.a = pk.y; else if (lane == 2) v = hm[j].x; else v = hm[j].y;
            vm_set_fp2(slots, VM_R_P2X + lane, v);
            zero = fp_is_zero(v.a) & fp_is_zero(v.b);
        }
        const unsigned zmask = __ballot_sync(0xffffffffu, zero);
        const bool skip = bad[j] != 0 || (zmask & 0x3) == 0x3 || (zmask & 0xc) == 0xc;
        if (skip) { if (lane == 0) atomicAdd(bad_count, 1u); __syncwarp(); continue; }
        vm_run(VM_P_ML1_INIT, slots);
        for (int i = 62; i >= 0; i--) {
            vm_run(VM_P_ML1_DBL, slots);
            if ((K_Z_ABS >> i) & 1) vm_run(VM_P_ML1_ADD, slots);
        }
        vm_run(VM_P_AMULF, slots);
    }
    if (lane < 12) vm_ld(reinterpret_cast<fp*>(&partial[6 * (size_t)blockIdx.x + (lane >> 1)])[lane & 1].l, slots, VM_R_A0 + (lane >> 1), lane & 1);
}
// product of W partial products (one warp)
__global__ void __launch_bounds__(32) k_rlc_reduce_coop(size_t W, const fp2* partial, fp2* out) {
    __shared__ uint32_t slots[VM_SMEM_WORDS];
    const int lane = threadIdx.x & 31;
    vm_load_consts(slots);
    vm_run(VM_P_A_ONE, slots);
    for (size_t w = 0; w < W; w++) {
        if (lane < 12) vm_st(slots, VM_R_F0 + (lane >> 1), lane & 1, reinterpret_cast<const fp*>(&partial[6 * w + (lane >> 1)])[lane & 1].l);
        __syncwarp();
        vm_run(VM_P_AMULF, slots);
    }
    if (lane < 12) vm_ld(reinterpret_cast<fp*>(&out[lane >> 1])[lane & 1].l, slots, VM_R_A0 + (lane >> 1), lane & 1);
}
// fold: verdict = FE( prod_p parts[p] * Miller(B, Sg) ) == 1, Sg = affine sum of the partial signature sums (not the identity)
__global__ void __launch_bounds__(32) k_rlc_fold_coop(size_t nparts, const fp2* parts, const g2a* Sg, uint8_t* result) {
    __shared__ uint32_t slots[VM_SMEM_WORDS];
    const int lane = threadIdx.x & 31;
    vm_load_consts(slots);
    vm_run(VM_P_A_ONE, slots);
    for (size_t w = 0; w < nparts; w++) {
        if (lane < 12) vm_st(slots, VM_R_F0 + (lane >> 1), lane & 1, reinterpret_cast<const fp*>(&parts[6 * w + (lane >> 1)])[lane & 1].l);
        __syncwarp();
        vm_run(VM_P_AMULF, slots);
    }
    bool zero = true;
    if (lane < 4) {
        fp2 v; fp2_zero(v);
        if (lane == 0) fp_set(v.a, K_G1_X); else if (lane == 1) fp_set(v.a, K_G1_Y); else if (lane == 2) v = Sg->x; else v = Sg->y;
        vm_set_fp2(slots, VM_R_P2X + lane, v);
        zero = fp_is_zero(v.a) & fp_is_zero(v.b);
    }
    const unsigned zmask = __ballot_sync(0xffffffffu, zero);
    if ((zmask & 0xc) == 0xc) { if (lane == 0) *result = 0; return; }       // empty / cancelling signature sum: not proven, callers fall back
    vm_run(VM_P_ML1_INIT, slots);
    for (int i = 62; i >= 0; i--) {
        vm_run(VM_P_ML1_DBL, slots);
        if ((K_Z_ABS >> i) & 1) vm_run(VM_P_ML1_ADD, slots);
    }
    vm_run(VM_P_FMULA, slots);
    const bool one = vm_final_exp_is_one(slots);
    if (lane == 0) *result = one ? 1 : 0;
}
// Jacobian G2 sum, single CTA (the partial signature sums)
__global__ void __launch_bounds__(HB_SUM_THREADS) k_g2_sum_jac(size_t n, const g2* in, g2* out) {
    __shared__ g2 sm[HB_SUM_THREADS];
    g2 acc; pt_set_inf(acc);
    for (size_t i = threadIdx.x; i < n; i += HB_SUM_THREADS) { g2 q = in[i]; pt_add(acc, acc, q); }
    sm[threadIdx.x] = acc;
    __syncthreads();
    for (int off = HB_SUM_THREADS / 2; off >= 1; off >>= 1) {
        if ((int)threadIdx.x < off) { g2 o = sm[threadIdx.x + off]; pt_add(acc, acc, o); sm[threadIdx.x] = acc; }
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = acc;
}

// ---- latency form, split in two: the Miller value of (B, sigma) only needs the decoded signature, so it is computed on the decode
// stream while hash-to-G2 (the long pole of a single check) still runs; the second kernel adds the pair (-apk, H(m)) and the final
// exponentiation.  f1: 6 Fp2 per round (tower order); irr1[j] = 1 when the signature is the identity / did not decode.
__global__ void __launch_bounds__(32) k_miller1_coop(size_t B, const g2a* sig, const uint8_t* ok_sig, fp2* f1, uint8_t* irr1) {
    __shared__ uint32_t slots[VM_SMEM_WORDS];
    const int lane = threadIdx.x & 31;
    vm_load_consts(slots);
    for (size_t j = blockIdx.x; j < B; j += gridDim.x) {
        bool zero = true;
        if (lane < 4) {
            fp2 v; fp2_zero(v);
            if (lane == 0) fp_set(v.a, K_G1_X); else if (lane == 1) fp_set(v.a, K_G1_Y); else if (lane == 2) v = sig[j].x; else v = sig[j].y;
            vm_set_fp2(slots, VM_R_P2X + lane, v);
            zero = fp_is_zero(v.a) & fp_is_zero(v.b);
        }
        const unsigned zmask = __ballot_sync(0xffffffffu, zero);
        const bool skip = (ok_sig && !ok_sig[j]) || (zmask & 0xc) == 0xc;
        if (lane == 0) irr1[j] = skip ? 1 : 0;
        if (skip) { __syncwarp(); continue; }
        vm_run(VM_P_ML1_INIT, slots);
        for (int i = 62; i >= 0; i--) {
            vm_run(VM_P_ML1_DBL, slots);
            if ((K_Z_ABS >> i) & 1) vm_run(VM_P_ML1_ADD, slots);
        }
        if (lane < 12) vm_ld(reinterpret_cast<fp*>(&f1[6 * j + (lane >> 1)])[lane & 1].l, slots, VM_R_F0 + (lane >> 1), lane & 1);
        __syncwarp();
    }
}
// ---- latency form with H(m) already known (the library's H(m) cache, hbls.cu): BOTH Miller values are independent of each other --
// (B, sigma) waits for the signature decode, (-apk, H(m)) only for the key aggregation -- so they run on two streams and a third
// kernel multiplies them and does the final exponentiation.  P = nullptr: the generator.  irr[j] = 1: an operand is the identity /
// did not decode (the round is then decided by k_pairing_fixup, like in the other forms).
__global__ void __launch_bounds__(32) k_miller_pq_coop(size_t B, const g1a* P, const g2a* Q, const uint8_t* ok_q, fp2* f, uint8_t* irr) {
    __shared__ uint32_t slots[VM_SMEM_WORDS];
    const int lane = threadIdx.x & 31;
    vm_load_consts(slots);
    for (size_t j = blockIdx.x; j < B; j += gridDim.x) {
        bool zero = true;
        if (lane < 4) {
            fp2 v; fp2_zero(v);
            if (lane < 2) { if (P) v.a = lane == 0 ? P[j].x : P[j].y; else fp_set(v.a, lane == 0 ? K_G1_X : K_G1_Y); }
            else v = lane == 2 ? Q[j].x : Q[j].y;
            vm_set_fp2(slots, VM_R_P2X + lane, v);
            zero = fp_is_zero(v.a) & fp_is_zero(v.b);
        }
        const unsigned zmask = __ballot_sync(0xffffffffu, zero);
        const bool skip = (ok_q && !ok_q[j]) || (zmask & 0x3) == 0x3 || (zmask & 0xc) == 0xc;
        if (lane == 0) irr[j] = skip ? 1 : 0;
        if (skip) { __syncwarp(); continue; }
        vm_run(VM_P_ML1_INIT, slots);
        for (int i = 62; i >= 0; i--) {
            vm_run(VM_P_ML1_DBL, slots);
            if ((K_Z_ABS >> i) & 1) vm_run(VM_P_ML1_ADD, slots);
        }
        if (lane < 12) vm_ld(reinterpret_cast<fp*>(&f[6 * j + (lane >> 1)])[lane & 1].l, slots, VM_R_F0 + (lane >> 1), lane & 1);
        __syncwarp();
    }
}
// verdict = FE(f1 f2) == 1; ok_sub (nullable): the signature's subgroup test, run beside its Miller loop
__global__ void __launch_bounds__(32) k_fe2_coop(size_t B, const fp2* f1, const uint8_t* irr1, const fp2* f2, const uint8_t* irr2,
                             const uint8_t* ok_a, const uint8_t* ok_b, const uint8_t* ok_c, const uint8_t* ok_sub, uint8_t* results) {
    __shared__ uint32_t slots[VM_SMEM_WORDS];
    const int lane = threadIdx.x & 31;
    vm_load_consts(slots);
    for (size_t j = blockIdx.x; j < B; j += gridDim.x) {
        const bool good = (!ok_a || ok_a[j]) && (!ok_b || ok_b[j]) && (!ok_c || ok_c[j]) && (!ok_sub || ok_sub[j]);
        const bool irregular = irr1[j] != 0 || irr2[j] != 0;
        bool one = false;
        if (!irregular) {
            if (lane < 12) {
                vm_st(slots, VM_R_A0 + (lane >> 1), lane & 1, reinterpret_cast<const fp*>(&f1[6 * j + (lane >> 1)])[lane & 1].l);
                vm_st(slots, VM_R_F0 + (lane >> 1), lane & 1, reinterpret_cast<const fp*>(&f2[6 * j + (lane >> 1)])[lane & 1].l);
            }
            __syncwarp();
            vm_run(VM_P_FMULA, slots);
            one = vm_final_exp_is_one(slots);
        }
        if (lane == 0) results[j] = irregular ? 0xFF : ((good && one) ? 1 : 0);
        __syncwarp();
    }
}
// subgroup test of already-decoded affine signatures, one item per lane pair (the second half of k_g2_decode_pair)
__global__ void k_g2_subgroup_pair(size_t n, const g2a* pts, const uint8_t* ok_in, uint8_t* ok_out) {
    const size_t i = HB_TID >> 1; if (i >= n) return;
    const g2a a = pts[i];
    bool good = ok_in[i] != 0;
    if (good && !aff_is_inf(a)) {
        jac<fp2h> q; fp2h_pack(q.x, a.x); fp2h_pack(q.y, a.y); fp2_one(q.z);
        good = g2_in_subgroup(q);
    }
    if ((threadIdx.x & 1) == 0) ok_out[i] = good ? 1 : 0;
}
__global__ void __launch_bounds__(32) k_pairing_coop2(size_t B, const fp2* f1, const uint8_t* irr1, const g1a* pk_neg, const g2a* hm,
                                  const uint8_t* ok_a, const uint8_t* ok_b, const uint8_t* ok_c, uint8_t* results) {
    __shared__ uint32_t slots[VM_SMEM_WORDS];
    const int lane = threadIdx.x & 31;
    vm_load_consts(slots);
    for (size_t j = blockIdx.x; j < B; j += gridDim.x) {
        const bool good = (!ok_a || ok_a[j]) && (!ok_b || ok_b[j]) && (!ok_c || ok_c[j]);
        bool zero = true;
        if (lane < 4) {
            fp2 v; fp2_zero(v);
            const g1a pk = pk_neg[j];
            if (lane == 0) v.a = pk.x; else if (lane == 1) v.a = pk.y; else if (lane == 2) v = hm[j].x; else v = hm[j].y;
            vm_set_fp2(slots, VM_R_P2X + lane, v);
            zero = fp_is_zero(v.a) & fp_is_zero(v.b);
        }
        const unsigned zmask = __ballot_sync(0xffffffffu, zero);
        const bool irregular = irr1[j] != 0 || (zmask & 0x3) == 0x3 || (zmask & 0xc) == 0xc;
        bool one = false;
        if (!irregular) {
            if (lane < 12) vm_st(slots, VM_R_A0 + (lane >> 1), lane & 1, reinterpret_cast<const fp*>(&f1[6 * j + (lane >> 1)])[lane & 1].l);
            __syncwarp();
            vm_run(VM_P_ML1_INIT, slots);
            for (int i = 62; i >= 0; i--) {
                vm_run(VM_P_ML1_DBL, slots);
                if ((K_Z_ABS >> i) & 1) vm_run(VM_P_ML1_ADD, slots);
            }
            vm_run(VM_P_FMULA, slots);
            one = vm_final_exp_is_one(slots);
        }
        if (lane == 0) results[j] = irregular ? 0xFF : ((good && one) ? 1 : 0);
        __syncwarp();
    }
}

// ------------------------------------------------------------------ random-linear-combination batch (R9 / R10 GPU form)
// prod_j [ e(B, sigma_j) e(-apk_j, H_j) ]^{r_j} == 1 with 64-bit r_j: the G rounds of a group share ONE Miller accumulator
// (pairs (-r_j apk_j, H_j) plus (B, sum_j r_j sigma_j)) and ONE final exponentiation.  The rounds of a group that fails -- or
// holds a round that did not decode -- are re-verified exactly afterwards (compacted list, k_pairing_verify_split_list), so
// results stay exact booleans (a bad round survives the batched test with probability <= 2^-63).
#ifndef HB_RLC_G
#define HB_RLC_G 4       // smallest group size (scratch is sized for it); the host picks 4 or 8 per call (hbls.cu).  At 75 776 rounds/step the
                         // pairing stage measured 76 / 48 / 68 / 65 ms for G = 3 / 4 / 5 / 7: the group count must still fill the SMs
#endif
#define HB_RLC_GMAX 8
// Groups are STRIDED: group g = rounds {g, g + ng, g + 2 ng, ...}; the coefficient depends only on the position k inside the
// group (c[k], fresh per call from the host's keyed ChaCha20 stream: hbls.cu rlc_draw), so the 32 consecutive rounds of a warp
// share one scalar and the double-and-add ladders run without divergence.  Sharing c[k] across groups is sound: every group's
// test passes wrongly with probability <= 2^-63 over the draw, whatever the (non-adaptive) input.
struct rlc_coeffs { uint64_t c[HB_RLC_GMAX]; };
// per round: P_j = -r_j apk_j (affine), S_j = r_j sigma_j (Jacobian), bad_j
#ifndef HB_SCALE_MINBLOCKS
#define HB_SCALE_MINBLOCKS 1
#endif
__global__ void __launch_bounds__(64, HB_SCALE_MINBLOCKS) k_rlc_scale(size_t B, size_t ng, const g1* apk, const g2a* sig, const g2a* hm, const uint8_t* ok_sig, const uint8_t* ok_hm,
                            const uint8_t* ok_pk, rlc_coeffs co, const uint64_t* per_item, g1a* pk_scaled_neg, g2* S, uint8_t* bad) {
  // per_item (nullable): one independent coefficient per round -- needed when ALL rounds enter one combined check (the split of a
  // single batch over several GPUs, k_rlc_partial_coop); the grouped form shares co.c[position in group] across groups
#if HB_BATCH_INV
  for (size_t j0 = HB_TID; j0 < B; j0 += (size_t)HB_BATCH_K * HB_STRIDE) {
    g1 ra[HB_BATCH_K]; fp z[HB_BATCH_K]; bool skip[HB_BATCH_K];
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t j = j0 + (size_t)k * HB_STRIDE;
        skip[k] = true;
        if (j >= B) continue;
        // grouped form: the FIRST round of every group keeps coefficient 1 (no ladders at all: a warp-uniform branch, since the 32
        // rounds of a warp share their position).  Sound: a group holding a bad round passes only if prod_j delta_j^{s_j} = 1 with
        // some delta_j != 1; if that j is 0 alone the product is delta_0 != 1, otherwise one of the random s_j (j >= 1) must hit
        // the single value mod r that cancels the rest -- probability <= 2^-63, as before.
        const uint64_t r = per_item ? per_item[j] : (j < ng ? 1ull : co.c[j / ng]);
        g1 a = apk[j]; g2a sg = sig[j]; g2a h = hm[j];
        const bool b = !ok_sig[j] || !ok_hm[j] || (ok_pk && !ok_pk[j]) || pt_is_inf(a) || aff_is_inf(sg) || aff_is_inf(h);
        g2 rs;
        if (r == 1ull && !per_item) { ra[k] = a; pt_from_aff(rs, sg); } else rlc_scale_pair(ra[k], rs, a, sg, r);
        S[j] = rs; bad[j] = b ? 1 : 0;
        skip[k] = pt_is_inf(ra[k]);
        if (!skip[k]) z[k] = ra[k].z;
    }
    f_batch_inv<fp, HB_BATCH_K>(z, skip);
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t j = j0 + (size_t)k * HB_STRIDE;
        if (j >= B) continue;
        g1a pa;
        if (skip[k]) { fp_zero(pa.x); fp_zero(pa.y); } else { pt_to_aff_zinv(pa, ra[k], z[k]); fp_neg(pa.y, pa.y); }
        pk_scaled_neg[j] = pa;
    }
  }
#else
  for (size_t j = HB_TID; j < B; j += HB_STRIDE) {
    const uint64_t r = per_item ? per_item[j] : (j < ng ? 1ull : co.c[j / ng]);
    g1 a = apk[j]; g2a sg = sig[j]; g2a h = hm[j];
    const bool b = !ok_sig[j] || !ok_hm[j] || (ok_pk && !ok_pk[j]) || pt_is_inf(a) || aff_is_inf(sg) || aff_is_inf(h);
    g1 ra; g2 rs;
    if (r == 1ull && !per_item) { ra = a; pt_from_aff(rs, sg); } else rlc_scale_pair(ra, rs, a, sg, r);
    g1a pa; pt_to_aff(pa, ra); fp_neg(pa.y, pa.y);
    pk_scaled_neg[j] = pa; S[j] = rs; bad[j] = b ? 1 : 0;
  }
#endif
}
// the same stage as two kernels, one ladder each (hbls.cu "scale_split"): the G1 ladder (+ shared-inversion affine conversion) and the
// G2 ladder are different code over different fields -- ncu on the fused kernel: stall_no_instruction 1.3 per issue
__global__ void k_rlc_scale_g1(size_t B, size_t ng, const g1* apk, rlc_coeffs co, g1a* pk_scaled_neg) {
  for (size_t j0 = HB_TID; j0 < B; j0 += (size_t)HB_BATCH_K * HB_STRIDE) {
    g1 ra[HB_BATCH_K]; fp z[HB_BATCH_K]; bool skip[HB_BATCH_K];
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t j = j0 + (size_t)k * HB_STRIDE;
        skip[k] = true;
        if (j >= B) continue;
        const g1 a = apk[j];
        if (j < ng) ra[k] = a; else rlc_scale_g1(ra[k], a, co.c[j / ng]);
        skip[k] = pt_is_inf(ra[k]);
        if (!skip[k]) z[k] = ra[k].z;
    }
    f_batch_inv<fp, HB_BATCH_K>(z, skip);
    for (int k = 0; k < HB_BATCH_K; k++) {
        const size_t j = j0 + (size_t)k * HB_STRIDE;
        if (j >= B) continue;
        g1a pa;
        if (skip[k]) { fp_zero(pa.x); fp_zero(pa.y); } else { pt_to_aff_zinv(pa, ra[k], z[k]); fp_neg(pa.y, pa.y); }
        pk_scaled_neg[j] = pa;
    }
  }
}
#ifndef HB_SCALE_G2_MINBLOCKS
#define HB_SCALE_G2_MINBLOCKS 1
#endif
__global__ void __launch_bounds__(64, HB_SCALE_G2_MINBLOCKS) k_rlc_scale_g2(size_t B, size_t ng, const g1* apk, const g2a* sig, const g2a* hm, const uint8_t* ok_sig, const uint8_t* ok_hm,
                               const uint8_t* ok_pk, rlc_coeffs co, g2* S, uint8_t* bad) {
  for (size_t j = HB_TID; j < B; j += HB_STRIDE) {
    const g2a sg = sig[j];
    const bool b = !ok_sig[j] || !ok_hm[j] || (ok_pk && !ok_pk[j]) || fp_is_zero(apk[j].z) || aff_is_inf(sg) || aff_is_inf(hm[j]);
    g2 rs;
    if (j < ng) pt_from_aff(rs, sg); else rlc_scale_g2(rs, sg, co.c[j / ng]);
    S[j] = rs; bad[j] = b ? 1 : 0;
  }
}
// per group: affine sum of its S_j
template <int G> __global__ void k_rlc_group_sum(size_t ngroups, const g2* S, g2a* Sg) {
  for (size_t g = HB_TID; g < ngroups; g += HB_STRIDE) {
    g2 acc; pt_set_inf(acc);
    for (int k = 0; k < G; k++) { g2 t = S[(size_t)k * ngroups + g]; pt_add(acc, acc, t); }
    g2a a; pt_to_aff(a, acc); Sg[g] = a;
  }
}
#ifndef HB_SMEM_F
#define HB_SMEM_F 0       // 1: keep each lane's Fp12 accumulator in dynamic shared memory (experiment: profiles/r2_stage_times.txt)
#endif
#define HB_SMEM_F_WORDS 73
// lane pair per group: (G + 1)-pair Miller loop, final exponentiation, verdict
template <int G> __global__ void __launch_bounds__(HB_TPB_SPLIT, HB_MINBLOCKS_SPLIT) k_rlc_pairing_split(size_t ngroups, const g1a* pk_scaled_neg, const g2a* hm, const g2a* Sg,
                                 const uint8_t* bad, uint8_t* group_ok) {
    const int role = threadIdx.x & 1;
    const size_t ppg = HB_STRIDE >> 1;
    __shared__ g1a gen_sh;
    if (threadIdx.x == 0) { fp_set(gen_sh.x, K_G1_X); fp_set(gen_sh.y, K_G1_Y); }
    __syncthreads();
    for (size_t it = 0; ; it++) {
        const size_t warp_first = it * ppg + ((HB_TID & ~(size_t)31) >> 1);
        if (warp_first >= ngroups) break;
        const size_t g = it * ppg + (HB_TID >> 1);
        const bool valid = g < ngroups;
        const size_t gg = valid ? g : ngroups - 1;
        const g1a* ps[G + 1]; fp2h qx[G + 1], qy[G + 1];
        bool anybad = false;
        for (int k = 0; k < G; k++) {
            const size_t j = (size_t)k * ngroups + gg;
            ps[k] = &pk_scaled_neg[j];
            const fp* h4 = reinterpret_cast<const fp*>(&hm[j]);
            qx[k].c = h4[role]; qy[k].c = h4[2 + role];
            anybad |= bad[j] != 0;
        }
        ps[G] = &gen_sh;
        const fp* s4 = reinterpret_cast<const fp*>(&Sg[gg]);
        qx[G].c = s4[role]; qy[G].c = s4[2 + role];
#if HB_SMEM_F
        // the Miller accumulator / exponentiation value of this lane in shared memory (73-word stride: conflict-free), not on the stack
        extern __shared__ uint32_t hb_dyn_smem[];
        fp12_t<fp2h>& m = *reinterpret_cast<fp12_t<fp2h>*>(hb_dyn_smem + (size_t)threadIdx.x * HB_SMEM_F_WORDS);
#else
        fp12_t<fp2h> m;
#endif
        miller_loop_multi<fp2h, G + 1>(m, ps, qx, qy);
        final_exp(m, m);
        const bool one = fp12_is_one(m);
        if (valid && role == 0) group_ok[g] = (one && !anybad) ? 1 : 0;
    }
}
// ---- the same check in TWO kernels (hbls.cu "rlc_two_phase").  The fused kernel above keeps G + 1 running points, the Fp12 accumulator
// and their temporaries per lane pair (4.5 KB of local memory per thread: 340 MB per launch, more than L2 -- ncu: 148 GB of DRAM traffic).
// Here the running points live in their OWN kernel: k_rlc_lines_split walks ONE pair (P, Q) per lane pair through the 63 doubling and
// 5 addition steps and writes the 68 line functions, already evaluated at P, to HBM (3 Fp2 per step: 19.6 KB per pair, read once);
// k_rlc_accum_split keeps only the accumulator: f <- f^2 * prod_k line_k per iteration, then the final exponentiation.
// Line layout: fp index ((step * 3 + c) * npairs + p) * 2 + role, p = k * ngroups + g: a warp's 32 lanes touch 1.5 KB contiguously.
#define HB_ML_STEPS 68                 // 63 doublings + 5 additions (bits 62, 60, 57, 48, 16 of |z|)
// the lines are written once and read once: streaming (evict-first) accesses keep them from pushing the kernels' own temporaries
// (local memory, which lives in L1 / L2) out of L2.  fp = 48 bytes at 16-byte aligned offsets: three 128-bit accesses.
HB_DEV void line_store(fp* dst, const fp& v) {
#ifdef HB_HOST_EMU
    *dst = v;
#else
    uint4* d = reinterpret_cast<uint4*>(dst);
    __stcs(d, make_uint4(v.l[0], v.l[1], v.l[2], v.l[3])); __stcs(d + 1, make_uint4(v.l[4], v.l[5], v.l[6], v.l[7])); __stcs(d + 2, make_uint4(v.l[8], v.l[9], v.l[10], v.l[11]));
#endif
}
HB_DEV void line_load(fp& v, const fp* src) {
#ifdef HB_HOST_EMU
    v = *src;
#else
    const uint4* s = reinterpret_cast<const uint4*>(src);
    const uint4 a = __ldcs(s), b = __ldcs(s + 1), c = __ldcs(s + 2);
    v.l[0] = a.x; v.l[1] = a.y; v.l[2] = a.z; v.l[3] = a.w; v.l[4] = b.x; v.l[5] = b.y; v.l[6] = b.z; v.l[7] = b.w; v.l[8] = c.x; v.l[9] = c.y; v.l[10] = c.z; v.l[11] = c.w;
#endif
}
template <int G> __global__ void __launch_bounds__(HB_TPB_SPLIT, HB_MINBLOCKS_SPLIT) k_rlc_lines_split(size_t ngtot, size_t g0, size_t ngroups, const g1a* pk_scaled_neg, const g2a* hm,
                                 const g2a* Sg, fp* lines, const unsigned* count = nullptr) {
    // groups g0 .. g0 + ngroups - 1 of ngtot (a chunk: the line buffer is sized for <= 37 888 groups); round of (k, g) = k * ngtot + g
    // count (nullable): the number of groups is only known on the device (compacted list of the failed groups' rounds)
    if (count) { const size_t n = *count; if (g0 >= n) return; ngtot = n; ngroups = n - g0 < ngroups ? n - g0 : ngroups; }
    const int role = threadIdx.x & 1;
    const size_t ppg = HB_STRIDE >> 1, npairs = (size_t)(G + 1) * ngroups;
    for (size_t it = 0; ; it++) {
        const size_t warp_first = it * ppg + ((HB_TID & ~(size_t)31) >> 1);
        if (warp_first >= npairs) break;
        const size_t p = it * ppg + (HB_TID >> 1);
        const bool valid = p < npairs;
        const size_t pp = valid ? p : npairs - 1, k = pp / ngroups, g = pp - k * ngroups;
        g1a P; const fp* q4;
        if (k < (size_t)G) { P = pk_scaled_neg[k * ngtot + g0 + g]; q4 = reinterpret_cast<const fp*>(&hm[k * ngtot + g0 + g]); }
        else { fp_set(P.x, K_G1_X); fp_set(P.y, K_G1_Y); q4 = reinterpret_cast<const fp*>(&Sg[g0 + g]); }
        fp2h qx, qy; qx.c = q4[role]; qy.c = q4[2 + role];
        g2proj_t<fp2h> T; T.x = qx; T.y = qy; fp2_one(T.z);
        fp2h l0, l2, l3;
        size_t st = 0;
        for (int i = 62; i >= 0; i--) {
#ifndef HB_LINES_SYNC
#define HB_LINES_SYNC 1
#endif
            if (HB_LINES_SYNC) hb_lockstep<fp2h>();
            ml_dbl(T, l0, l2, l3); fp2_mul_fp(l2, l2, P.x); fp2_mul_fp(l3, l3, P.y);
            if (valid) { fp* o = lines + ((st * 3) * npairs + pp) * 2 + role; line_store(o, l0.c); line_store(o + 2 * npairs, l2.c); line_store(o + 4 * npairs, l3.c); }
            st++;
            if ((K_Z_ABS >> i) & 1) {
                ml_add(T, qx, qy, l0, l2, l3); fp2_mul_fp(l2, l2, P.x); fp2_mul_fp(l3, l3, P.y);
                if (valid) { fp* o = lines + ((st * 3) * npairs + pp) * 2 + role; line_store(o, l0.c); line_store(o + 2 * npairs, l2.c); line_store(o + 4 * npairs, l3.c); }
                st++;
            }
        }
    }
}
template <int G> __global__ void __launch_bounds__(HB_TPB_SPLIT, HB_MINBLOCKS_SPLIT) k_rlc_accum_split(size_t ngtot, size_t g0, size_t ngroups, const fp* lines, const uint8_t* bad, uint8_t* group_ok, const unsigned* count = nullptr) {
    if (count) { const size_t n = *count; if (g0 >= n) return; ngtot = n; ngroups = n - g0 < ngroups ? n - g0 : ngroups; }
    const int role = threadIdx.x & 1;
    const size_t ppg = HB_STRIDE >> 1, npairs = (size_t)(G + 1) * ngroups;
    for (size_t it = 0; ; it++) {
        const size_t warp_first = it * ppg + ((HB_TID & ~(size_t)31) >> 1);
        if (warp_first >= ngroups) break;
        const size_t g = it * ppg + (HB_TID >> 1);
        const bool valid = g < ngroups;
        const size_t gg = valid ? g : ngroups - 1;
        bool anybad = false;
        for (int k = 0; k < G; k++) anybad |= bad[(size_t)k * ngtot + g0 + gg] != 0;
        fp12_t<fp2h> m; fp12_one(m);
        size_t st = 0;
#ifndef HB_LINE_PAIRS
#define HB_LINE_PAIRS 0          // 1: lines are multiplied two by two before they touch the accumulator (23 instead of 26 Fp2 products):
#endif                           // measured 99.1 vs 96.9 ms -- the extra temporaries cost more than the 10 % fewer products save
#ifndef HB_ACCUM_SYNC
#define HB_ACCUM_SYNC 0          // CTA re-alignment every this many lines inside an iteration (0: only once per iteration, -1: never);
                                 // measured (pairing stage, 303 104 rounds): every 2 lines 98.5, every 4 96.9, per iteration only 95.7, never 100.5 ms
#endif
        auto mul_lines = [&](size_t step) {
            const fp* base = lines + ((step * 3) * npairs + gg) * 2 + role;
#pragma unroll 1
            for (int k = 0; k <= G; k += HB_LINE_PAIRS ? 2 : 1) {
                if (HB_ACCUM_SYNC > 0 && G > 4 && (k % (HB_ACCUM_SYNC > 0 ? HB_ACCUM_SYNC : 1)) == 0 && k) hb_lockstep<fp2h>();
                const fp* o = base + (size_t)k * ngroups * 2;
                fp2h l0, l2, l3; line_load(l0.c, o); line_load(l2.c, o + 2 * npairs); line_load(l3.c, o + 4 * npairs);
                if (HB_LINE_PAIRS && k + 1 <= G) {
                    const fp* o2 = o + ngroups * 2;
                    fp2h n0, n2, n3; line_load(n0.c, o2); line_load(n2.c, o2 + 2 * npairs); line_load(n3.c, o2 + 4 * npairs);
                    fp12_mul_by_two_lines(m, m, l0, l2, l3, n0, n2, n3);
                } else
                    fp12_mul_by_014(m, m, l0, l2, l3);
            }
        };
        for (int i = 62; i >= 0; i--) {
            if (HB_ACCUM_SYNC >= 0) hb_lockstep<fp2h>();
            fp12_sqr(m, m);
            mul_lines(st++);
            if ((K_Z_ABS >> i) & 1) mul_lines(st++);
        }
        final_exp(m, m);
        const bool one = fp12_is_one(m);
        if (valid && role == 0) group_ok[g0 + g] = (one && !anybad) ? 1 : 0;
    }
}
// ---- the EXACT check through the same two kernels: a "group" of ONE round = the pairs (-apk_j, H(m_j)) and (B, sigma_j), i.e.
// k_rlc_lines_split<1> / k_rlc_accum_split<1> with pk_scaled_neg = -apk (affine) and Sg = the decoded signatures.  These two small
// kernels prepare the flags (a round with an identity operand is left to k_pairing_fixup: 0xFF, as in k_pairing_verify_split)
// and publish the verdicts.  idx (nullable): the rounds are those of a compacted list (failed groups of the batched form).
__global__ void k_exact_prepare(size_t n, const uint32_t* idx, const g2a* sig, const g1a* pk_neg, const g2a* hm, const uint8_t* ok_a, const uint8_t* ok_b,
                                const uint8_t* ok_c, g1a* pk_c, g2a* hm_c, g2a* sig_c, uint8_t* bad, uint8_t* results, const unsigned* count = nullptr) {
    if (count) n = *count;
    const size_t t = HB_TID; if (t >= n) return;
    const size_t j = idx ? idx[t] : t;
    const g2a s = sig[j], h = hm[j]; const g1a p = pk_neg[j];
    const bool good = (!ok_a || ok_a[j]) && (!ok_b || ok_b[j]) && (!ok_c || ok_c[j]);
    const bool irregular = aff_is_inf(s) || aff_is_inf(h) || aff_is_inf(p);
    bad[t] = (!good || irregular) ? 1 : 0;
    if (pk_c) { pk_c[t] = p; hm_c[t] = h; sig_c[t] = s; }               // gathered copies (list form)
    results[j] = irregular ? 0xFF : 0;
}
__global__ void k_exact_publish(size_t n, const uint32_t* idx, const uint8_t* verdict, uint8_t* results, const unsigned* count = nullptr) {
    if (count) n = *count;
    const size_t t = HB_TID; if (t >= n) return;
    const size_t j = idx ? idx[t] : t;
    if (results[j] != 0xFF) results[j] = verdict[t];
}
// verdicts of the groups -> per-round results; the rounds of failed groups are compacted into `list` for the exact pass.
// counts[0] = rounds listed, counts[1] = groups that failed (hbls_last_batch_info)
__global__ void k_rlc_finish(size_t nrounds, size_t ngroups, const uint8_t* group_ok, uint8_t* results, uint32_t* list, unsigned* counts) {
    size_t j = HB_TID; if (j >= nrounds) return;
    const uint8_t ok = group_ok[j % ngroups];
    results[j] = ok;
    if (!ok) {
        list[atomicAdd(&counts[0], 1u)] = (uint32_t)j;
        if (j < ngroups) atomicAdd(&counts[1], 1u);
    }
}
__global__ void k_g1_normalize_list(const unsigned* count, const uint32_t* list, const g1* in, g1a* out, int negate) {
  const size_t n = *count;
  for (size_t i = HB_TID; i < n; i += HB_STRIDE) {
    const size_t j = list[i];
    g1 p = in[j]; g1a a; pt_to_aff(a, p);
    if (negate) fp_neg(a.y, a.y);
    out[j] = a;
  }
}
// k_pairing_verify_split over the listed rounds only (same body, indirect round index)
__global__ void __launch_bounds__(HB_TPB_SPLIT, HB_MINBLOCKS_SPLIT) k_pairing_verify_split_list(const unsigned* count, const uint32_t* list, const g2a* sig, const g1a* pk_neg,
                                 const g2a* hm, const uint8_t* ok_a, const uint8_t* ok_b, const uint8_t* ok_c, uint8_t* results) {
    const size_t B = *count;
    if (B == 0) return;
    const int role = threadIdx.x & 1;
    const size_t ppg = HB_STRIDE >> 1;
    for (size_t it = 0; ; it++) {
        const size_t warp_first = it * ppg + ((HB_TID & ~(size_t)31) >> 1);
        if (warp_first >= B) break;
        const size_t i = it * ppg + (HB_TID >> 1);
        const bool valid = i < B;
        const size_t jj = list[valid ? i : B - 1];
        bool good = (!ok_a || ok_a[jj]) && (!ok_b || ok_b[jj]) && (!ok_c || ok_c[jj]);
        g1a gen, p2 = pk_neg[jj];
        fp_set(gen.x, K_G1_X); fp_set(gen.y, K_G1_Y);
        const fp* s4 = reinterpret_cast<const fp*>(&sig[jj]);
        const fp* h4 = reinterpret_cast<const fp*>(&hm[jj]);
        fp2h q1x, q1y, q2x, q2y;
        q1x.c = s4[role]; q1y.c = s4[2 + role]; q2x.c = h4[role]; q2y.c = h4[2 + role];
        const bool z1x = fp2_is_zero(q1x), z1y = fp2_is_zero(q1y), z2x = fp2_is_zero(q2x), z2y = fp2_is_zero(q2y);
        const bool irregular = (z1x & z1y) | (z2x & z2y) | (fp_is_zero(p2.x) & fp_is_zero(p2.y));
        fp12_t<fp2h> m;
        miller_loop2<fp2h>(m, gen, q1x, q1y, p2, q2x, q2y, true, true);
        final_exp(m, m);
        const bool one = fp12_is_one(m);
        if (valid && role == 0) results[jj] = irregular ? 0xFF : ((good && one) ? 1 : 0);
    }
}
__global__ void k_pairing_fixup_list(const unsigned* count, const uint32_t* list, const g2a* sig, const g1a* pk_neg, const g2a* hm,
                                     const uint8_t* ok_a, const uint8_t* ok_b, const uint8_t* ok_c, uint8_t* results) {
  const size_t n = *count;
  for (size_t i = HB_TID; i < n; i += HB_STRIDE) {
    const size_t j = list[i];
    if (results[j] != 0xFF) continue;
    bool good = (!ok_a || ok_a[j]) && (!ok_b || ok_b[j]) && (!ok_c || ok_c[j]);
    g1a gen, p2 = pk_neg[j]; g2a q1 = sig[j], q2 = hm[j];
    fp_set(gen.x, K_G1_X); fp_set(gen.y, K_G1_Y);
    results[j] = (good && verify_irregular(gen, q1, p2, q2)) ? 1 : 0;
  }
}
// headers / items callers want to tell "signature bytes do not decode" from "pairing check failed" (engine.go:630-640 returns
// different errors): flags[j] bit0 = signature decoded, bit1 = message mapped to a point, bit2 = public key decoded
__global__ void k_pack_flags(size_t n, const uint8_t* ok_sig, const uint8_t* ok_hm, const uint8_t* ok_pk, uint8_t* flags) {
    size_t j = HB_TID; if (j >= n) return;
    flags[j] = (ok_sig[j] ? 1 : 0) | (ok_hm[j] ? 2 : 0) | ((!ok_pk || ok_pk[j]) ? 4 : 0);
}

// device self-test of the lane-pair Fp2 primitives against the single-thread ones on pseudo-random operands
__global__ void k_selftest_fp2h(uint32_t n, uint32_t seed, uint32_t* mismatches) {
    const int role = threadIdx.x & 1;
    for (uint32_t it = 0; it < n; it++) {
        uint32_t st = seed + 7919u * (uint32_t)(HB_TID >> 1) + 104729u * it;
        fp2 x, y;
        uint32_t* w[4] = {x.a.l, x.b.l, y.a.l, y.b.l};
        for (int c = 0; c < 4; c++) { for (int k = 0; k < 12; k++) { st = st * 1664525u + 1013904223u; w[c][k] = st ^ (st >> 13); } w[c][11] &= 0x0fffffffu; }
        fp2h hx, hy, hr; hx.c = role ? x.b : x.a; hy.c = role ? y.b : y.a;
        fp2 r; uint32_t bad = 0;
#define HB_CHK() do { const fp& e = role ? r.b : r.a; if (!fp_eq(e, hr.c)) bad++; } while (0)
        fp2_mul(r, x, y); fp2_mul(hr, hx, hy); HB_CHK();
        fp2_sqr(r, x); fp2_sqr(hr, hx); HB_CHK();
        fp2_mul_xi(r, x); fp2_mul_xi(hr, hx); HB_CHK();
        fp2_conj(r, y); fp2_conj(hr, hy); HB_CHK();
        fp2_add(r, x, y); fp2_add(hr, hx, hy); HB_CHK();
        fp2_sub(r, x, y); fp2_sub(hr, hx, hy); HB_CHK();
        fp2_neg(r, x); fp2_neg(hr, hx); HB_CHK();
        fp2_dbl(r, y); fp2_dbl(hr, hy); HB_CHK();
        fp2_mul_fp(r, x, y.a); fp2_mul_fp(hr, hx, y.a); HB_CHK();
        fp2_inv(r, x); fp2_inv(hr, hx); HB_CHK();
        fp2_one(r); fp2_one(hr); HB_CHK();
        fp2_const(r, K_PSI_CX); fp2_const(hr, K_PSI_CX); HB_CHK();
        if (fp2_is_zero(hx) != fp2_is_zero(x)) bad++;
        fp2 z; fp2_zero(z); fp2h hz; fp2_zero(hz); if (!fp2_is_zero(hz)) bad++;
        if (bad) atomicAdd(mismatches, bad);
    }
}

// ---- scalar multiplication batches (R6 sign, R14 GetPublicKey)
__global__ void k_g1_mul_gen(size_t n, const uint8_t* sk32, g1* out) {
    size_t i = HB_TID; if (i >= n) return;
    uint32_t k[8]; load_words(k, sk32 + 32 * i, 8);
    g1 g, r; g1_generator(g); pt_mul(r, g, k, 8); out[i] = r;
}
__global__ void k_sign_hash(size_t n, const uint8_t* sk32, const uint8_t* msgs, uint32_t msg_len, g2* out, uint8_t* ok) {
    size_t i = HB_TID; if (i >= n) return;
    uint32_t k[8]; load_words(k, sk32 + 32 * i, 8);
    g2 h, r; bool good = map_to_g2(h, msgs + (size_t)msg_len * i, msg_len);
    if (good) pt_mul(r, h, k, 8); else pt_set_inf(r);
    out[i] = r; ok[i] = good ? 1 : 0;
}
// sigma = sk * H for an already-mapped H(m) (the library's H(m) cache, hbls.cu): one item per LANE PAIR, the 255-bit ladder on the
// split carrier.  hm_stride = 0: every item signs the same point.  Output Jacobian (the layout of blsSignature).
__global__ void k_sign_hm_pair(size_t n, const uint8_t* sk32, const g2a* hm, const uint8_t* ok_hm, size_t hm_stride, g2* out, uint8_t* ok) {
    const size_t i = HB_TID >> 1; if (i >= n) return;
    uint32_t k[8]; load_words(k, sk32 + 32 * i, 8);
    const g2a h = hm[i * hm_stride];
    const bool good = ok_hm[i * hm_stride] != 0 && !aff_is_inf(h);
    jac<fp2h> H, R; fp2h_pack(H.x, h.x); fp2h_pack(H.y, h.y); fp2_one(H.z);
    pt_mul(R, H, k, 8);
    g2 r; fp2h_unpack(r.x, R.x); fp2h_unpack(r.y, R.y); fp2h_unpack(r.z, R.z);
    if (!good) pt_set_inf(r);
    if ((threadIdx.x & 1) == 0) { out[i] = r; ok[i] = good ? 1 : 0; }
}
// The same signature through the psi endomorphism (latency path of blsSignHash): the host writes sk = d0 + d1 Z + d2 Z^2 + d3 Z^3 in
// base Z = |z| (four 64-bit digits: sk < r < Z^4); on G2 psi acts as [z] = [-Z], so  sk H = d0 H - d1 psi(H) + d2 psi^2(H) - d3 psi^3(H)
// is ONE 64-step ladder over a 15-entry table of subset sums (64 doublings + <= 64 additions instead of 255 + 64 + 14).
__global__ void k_sign_hm_gls_pair(size_t n, const uint64_t* digits, const g2a* hm, const uint8_t* ok_hm, size_t hm_stride, g2* out, uint8_t* ok) {
    const size_t i = HB_TID >> 1; if (i >= n) return;
    const uint64_t d0 = digits[4 * i], d1 = digits[4 * i + 1], d2 = digits[4 * i + 2], d3 = digits[4 * i + 3];
    const g2a h = hm[i * hm_stride];
    const bool good = ok_hm[i * hm_stride] != 0 && !aff_is_inf(h);
    jac<fp2h> T[16], R;
    pt_set_inf(T[0]);
    fp2h_pack(T[1].x, h.x); fp2h_pack(T[1].y, h.y); fp2_one(T[1].z);          // H
    g2_psi(T[2], T[1]); pt_neg(T[2], T[2]);                                    // -psi(H)
    g2_psi2(T[4], T[1]);                                                       // psi^2(H)
    g2_psi(T[8], T[4]); pt_neg(T[8], T[8]);                                    // -psi^3(H)
    for (int m = 3; m < 16; m++) if (m & (m - 1)) pt_add(T[m], T[m & (m - 1)], T[m & -m]);
    pt_set_inf(R);
    for (int b = 63; b >= 0; b--) {
        pt_dbl(R, R);
        const int m = (int)((d0 >> b) & 1) | (int)((d1 >> b) & 1) << 1 | (int)((d2 >> b) & 1) << 2 | (int)((d3 >> b) & 1) << 3;
        if (m) pt_add(R, R, T[m]);
    }
    g2 r; fp2h_unpack(r.x, R.x); fp2h_unpack(r.y, R.y); fp2h_unpack(r.z, R.z);
    if (!good) pt_set_inf(r);
    if ((threadIdx.x & 1) == 0) { out[i] = r; ok[i] = good ? 1 : 0; }
}

// ---- single-element ops behind the herumi-shaped C ABI (one thread; latency is launch-bound)
// (Sign / PublicKey Deserialize run batched: k_g2_decode_pair with the struct epilogue, k_g1_decode_jac)
enum { OP_G1_ADD = 1, OP_G1_SUB, OP_G2_ADD, OP_G1_EQ, OP_G2_EQ, OP_G1_SER, OP_G2_SER, OP_MAP_SER, OP_G2_DES_ADD };
__global__ void k_single(int op, const void* a, const void* b, void* out, int* rc, uint32_t len) {
    if (HB_TID != 0) return;
    switch (op) {
    case OP_G1_ADD: case OP_G1_SUB: {
        g1 x = *(const g1*)a, y = *(const g1*)b; if (op == OP_G1_SUB) pt_neg(y, y);
        pt_add(x, x, y); *(g1*)out = x; *rc = 0; break; }
    case OP_G2_ADD: { g2 x = *(const g2*)a, y = *(const g2*)b; pt_add(x, x, y); *(g2*)out = x; *rc = 0; break; }
    case OP_G1_EQ: { g1 x = *(const g1*)a, y = *(const g1*)b; *rc = pt_eq(x, y) ? 1 : 0; break; }
    case OP_G2_EQ: { g2 x = *(const g2*)a, y = *(const g2*)b; *rc = pt_eq(x, y) ? 1 : 0; break; }
    case OP_G1_SER: { g1 x = *(const g1*)a; g1_serialize((uint8_t*)out, x); *rc = 48; break; }
    case OP_G2_SER: { g2 x = *(const g2*)a; g2_serialize((uint8_t*)out, x); *rc = 96; break; }
    case OP_MAP_SER: { g2 h; bool g = map_to_g2(h, (const uint8_t*)a, len); if (g) g2_serialize((uint8_t*)out, h); *rc = g ? 0 : -1; break; }
    case OP_G2_DES_ADD: {   // ballot box: out (Jacobian running sum) += decode(a); rc = 96 ok / 0 undecodable (sum untouched)
        g2 x; bool g = g2_deserialize(x, (const uint8_t*)a, true);
        if (g) { g2 acc = *(const g2*)out; pt_add(acc, acc, x); *(g2*)out = acc; }
        *rc = g ? 96 : 0; break; }
    default: *rc = -1;
    }
}

// ---- integer-pipe roofline probe: K independent accumulator sets per thread, each fed by lane_mad -- the exact
// mad.lo.cc / madc.hi.cc chains of the field multiplier (SASS: IMAD.WIDE.U32(.X), 6 per lane_mad).  Round 1 probed two loop
// invariants with a plain mad.wide; ptxas hoisted the product and the loop became IADD3 pairs, so the "18 TMAC32/s" it
// reported was half the ALU add rate.  Measured on B200 (tools/probe_int.cu, profiles/r2_probe_int.*): an IMAD.WIDE occupies the
// FMA-heavy pipe for 4 cycles per warp (a 32-bit IMAD for 2), i.e. 8 wide MACs per clock per scheduler.
template <int K> __global__ void k_probe_carry(int iters, uint32_t seed, uint32_t* sink, unsigned long long* cycles) {
    uint32_t acc[K][14], a[12];
    uint32_t t = seed ^ (uint32_t)HB_TID;
#pragma unroll
    for (int j = 0; j < 12; j++) { t = t * 1664525u + 1013904223u; a[j] = t; }
#pragma unroll
    for (int k = 0; k < K; k++)
#pragma unroll
        for (int j = 0; j < 14; j++) { t = t * 1664525u + 1013904223u; acc[k][j] = t; }
    const uint32_t b = t | 1u;
    const long long c0 = clock64();
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < K; k++) lane_mad(acc[k], a, b);
    }
    const long long c1 = clock64();
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < K; k++)
#pragma unroll
        for (int j = 0; j < 14; j++) s ^= acc[k][j];
    if (s == 0x12345u) sink[0] = s;                // never true in practice: keeps the chains alive
    if (HB_TID == 0) cycles[0] = (unsigned long long)(c1 - c0);
}

}  // namespace hb
