/*
 * include/hbls.h -- C ABI of libhbls.so, the B200-native (CUDA sm_100a) BLS12-381 backend for Harmony's
 * signature aggregation / aggregate-verification hot path.
 *
 * This is exactly what the reference's FFI for this path binds:
 *   - Part 1 mirrors the herumi `bls.h` subset that `github.com/harmony-one/bls/ffi/go/bls` (reference go.mod:27)
 *     calls through cgo, built with BLS_SWAP_G=1 (reference Makefile:68-70): public keys in G1 (48 B),
 *     signatures in G2 (96 B).  Every Go identifier the reference uses (SURVEY.md 8b) maps to one function here.
 *   - Part 2 are additive batch entry points that `crypto/bls` wrappers call so that a whole committee round /
 *     block range crosses cgo once (mask.go:113-134 SetMask, mask.go:58-64 AggregateSig,
 *     internal/chain/engine.go:619-642 verifySignature, consensus/leader.go:227-290 onCommit loop).
 *
 * Conventions: plain pointers and sizes only; all memory caller-owned; no callbacks; int error codes.
 * Threading: every function may be called from any thread after blsInit.  Concurrent per-call blsVerifyHash / blsVerify,
 * blsSignHash / blsSign, blsSignatureDeserialize, blsPublicKeyDeserialize and blsGetPublicKey calls are COALESCED: each queues its
 * request, and one of the waiting callers (no extra thread) takes the library mutex, drains up to coop_max queued requests and runs
 * them as one batched device pass per operation kind -- each caller gets exactly the result and output bytes of a lone call.  A
 * request waits at most for the batch in flight (or the batch call holding the mutex) and then leaves in the next batch; a lone
 * caller runs a batch of one at once.  Everything else -- Add / Sub / IsEqual / Serialize and the batch entry points of Part 2 --
 * runs one call at a time under the library mutex.  All of it runs on one library stream (except
 * hbls_aggregate_verify_batch_device on a caller stream).  Scratch memory is per stream, so asynchronous device-pointer calls on
 * DIFFERENT streams do not share intermediates; calls on one stream are stream-ordered.
 * Messages: only the first min(len, 48) bytes enter the map to G2 (mcl setArrayMask; SURVEY A.3); batch entry points take the
 * message stride msg_len and read min(msg_len, 48) bytes per item.
 * Identity operands: VerifyHash / aggregate-verify with an identity public key (e.g. an empty bitmap) returns 0 -- a zero key would
 * make the zero signature "valid" for every message.  (Unpinned by the reference's tests, SURVEY A.7; current herumi does the same.)
 * There is NO CPU fallback: if no CUDA device is usable blsInit returns HBLS_ERR_CUDA and every other call fails.
 */
#ifndef HBLS_H
#define HBLS_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define HBLS_BLS12_381 5            /* bls.BLS12_381 (crypto/bls/mask.go:18-20) */
#define HBLS_COMPILED_TIME_VAR 46   /* MCLBN_FR_UNIT_SIZE*10 + MCLBN_FP_UNIT_SIZE = 4*10 + 6 */

#define HBLS_ERR_CUDA   (-100)      /* no device / CUDA runtime failure (message on stderr) */
#define HBLS_ERR_ARG    (-2)        /* bad argument (e.g. bitmap length mismatch: mask.go:114-120) */
#define HBLS_ERR_DECODE (-3)        /* an input failed to decode (not on curve / >= p / not in subgroup) */

/* ------------------------------------------------------------------ Part 1: herumi bls.h shape (SWAP_G) */
typedef struct { uint64_t d[4]; }  blsSecretKey;   /* 32 B: scalar < r, little-endian */
typedef struct { uint64_t d[18]; } blsPublicKey;   /* 144 B: G1 Jacobian, Montgomery limbs; all-zero = identity */
typedef struct { uint64_t d[36]; } blsSignature;   /* 288 B: G2 Jacobian, Montgomery limbs; all-zero = identity */

/* bls.Init(bls.BLS12_381): crypto/bls/mask.go:18-20, internal/utils/utils.go:33.  0 = ok. */
int blsInit(int curve, int compiledTimeVar);
/* like blsInit but pins the CUDA device (one process per GPU: device = LOCAL_RANK) */
int hbls_init_device(int device);

/* SecretKey.SetByCSPRNG (crypto/bls/mask.go:23-27 RandPrivateKey) */
int blsSecretKeySetByCSPRNG(blsSecretKey* sec);
/* SecretKey.GetPublicKey: pk = sk * B, B = herumi SWAP_G generator (SURVEY A.2) */
void blsGetPublicKey(blsPublicKey* pub, const blsSecretKey* sec);
/* SecretKey.SignHash (consensus/construct.go:101,110): 0 ok, -1 when the message maps to no point */
int blsSignHash(blsSignature* sig, const blsSecretKey* sec, const void* h, size_t size);
/* Sign.VerifyHash (consensus/leader.go:173,287; internal/chain/engine.go:638): 1 valid, 0 invalid */
int blsVerifyHash(const blsSignature* sig, const blsPublicKey* pub, const void* h, size_t size);
/* SecretKey.Sign(string) / Sign.Verify(string): tests only, bytes unpinned by the reference (SURVEY A.7) */
void blsSign(blsSignature* sig, const blsSecretKey* sec, const void* m, size_t size);
int blsVerify(const blsSignature* sig, const blsPublicKey* pub, const void* m, size_t size);

/* PublicKey.Add / Sub (crypto/bls/mask.go:126,130), Sign.Add (mask.go:61).  The herumi signatures are void; a CUDA failure
 * leaves the destination as the identity and is reported by hbls_last_error(). */
void blsPublicKeyAdd(blsPublicKey* pub, const blsPublicKey* rhs);
void blsPublicKeySub(blsPublicKey* pub, const blsPublicKey* rhs);
void blsSignatureAdd(blsSignature* sig, const blsSignature* rhs);

/* Serialize: bytes written (32/48/96) or 0 on error.  Deserialize: bytes read or 0 on error
 * (>= p, not on curve, not in the r-torsion; scalar >= r). */
size_t blsSecretKeySerialize(void* buf, size_t maxBufSize, const blsSecretKey* sec);
size_t blsPublicKeySerialize(void* buf, size_t maxBufSize, const blsPublicKey* pub);
size_t blsSignatureSerialize(void* buf, size_t maxBufSize, const blsSignature* sig);
size_t blsSecretKeyDeserialize(blsSecretKey* sec, const void* buf, size_t bufSize);
size_t blsPublicKeyDeserialize(blsPublicKey* pub, const void* buf, size_t bufSize);
size_t blsSignatureDeserialize(blsSignature* sig, const void* buf, size_t bufSize);

/* PublicKey.GetAddress (internal/utils/utils.go:77, consensus/consensus_block_proposing.go:55): first 20 bytes of
 * SHA-256(Serialize(pub)).  Bytes unpinned by the reference's tests (SURVEY A.7).  0 ok. */
int hbls_get_address(const blsPublicKey* pub, uint8_t out20[20]);
/* last CUDA / runtime error seen by a call that cannot return one (the void Part-1 functions): returns the cudaError_t value
 * (0 = none) and clears it; msg (nullable) receives a short description */
int hbls_last_error(char* msg, size_t msg_cap);

int blsSecretKeyIsEqual(const blsSecretKey* lhs, const blsSecretKey* rhs);
int blsPublicKeyIsEqual(const blsPublicKey* lhs, const blsPublicKey* rhs);
int blsSignatureIsEqual(const blsSignature* lhs, const blsSignature* rhs);

/* ------------------------------------------------------------------ Part 2: batch entry points (device-resident committee) */
typedef struct hbls_committee hbls_committee;

/* Decode + subgroup-check n public keys once and keep the table in HBM (mirrors the epochCtx cache of
 * internal/chain/engine.go:644-659,727-761 and BLSPubKeyCache of crypto/bls/mask.go:35-55).
 * 0 ok; HBLS_ERR_DECODE if any key is invalid (*bad_index, if non-NULL, receives the first offender). */
int hbls_committee_create(hbls_committee** out, const uint8_t* pk48, size_t n, size_t* bad_index);
void hbls_committee_destroy(hbls_committee* c);
size_t hbls_committee_size(const hbls_committee* c);

/* Mask.SetMask on a fresh mask + AggregatePublic.Serialize (crypto/bls/mask.go:113-134).
 * bitmap: LSB-first within each byte; blen must equal (n+7)>>3 else HBLS_ERR_ARG. */
int hbls_mask_aggregate(const hbls_committee* c, const uint8_t* bitmap, size_t blen, uint8_t out_pk48[48]);

/* AggregateSig (crypto/bls/mask.go:58-64; consensus/quorum/quorum.go:164-196 AggregateVotes):
 * decode n signatures (with subgroup check) and sum them.  0 ok, HBLS_ERR_DECODE if one fails. */
int hbls_aggregate_sigs(const uint8_t* sig96, size_t n, uint8_t out96[96]);

/* FastAggregateVerify / VerifyAggregateSig of BASELINE.json == the reference composition
 * Deserialize(sig) ; SetMask(bitmap) ; aggSig.VerifyHash(mask.AggregatePublic, msg)
 * (internal/chain/engine.go:630-640, consensus/validator.go:219-236).  1 valid, 0 invalid, <0 error. */
int hbls_aggregate_verify(const hbls_committee* c, const uint8_t* bitmap, size_t blen,
                          const uint8_t sig96[96], const void* msg, size_t msg_len);

/* B independent rounds against one committee (block-range sync: api/service/stagedstreamsync/sig_verify.go:23-58).
 * bitmaps: B*blen bytes; sigs96: B*96; msgs: B*msg_len (msg_len <= 64); results[j] = 1/0. */
int hbls_aggregate_verify_batch(const hbls_committee* c, size_t B, const uint8_t* bitmaps, size_t blen,
                                const uint8_t* sigs96, const uint8_t* msgs, size_t msg_len, uint8_t* results);
/* How the batch entries check the pairing equations.
 * mode 1 (default): random-linear-combination groups -- 4 or 8 rounds share one Miller accumulator and one final exponentiation
 *   (prod_j [e(B, sigma_j) e(-apk_j, H_j)]^{r_j} == 1; r_j = a_j + b_j z^2 from a fresh 64-bit draw per group position and call out of
 *   a ChaCha20 stream keyed from /dev/urandom at blsInit).  The rounds of every group that fails or holds an undecodable round are
 *   re-verified exactly (those rounds only), so results are the exact booleans; a bad round survives the batched test with
 *   probability <= 2^-63.  Batches under `rlc_min` rounds (default 12 288, hbls_set_param) always use mode 0, and up to `coop_max`
 *   rounds the exact check runs one WARP per round (latency form, csrc/vm.cuh) instead of one lane pair.
 * mode 0: the exact per-round check only (identical semantics to N calls of hbls_aggregate_verify). */
void hbls_set_batch_mode(int mode);
int  hbls_get_batch_mode(void);
/* what the most recent batch call (aggregate_verify_batch[_device], verify_batch, aggregate_verify_items, verify_headers) did:
 * waits for that call's device work if it is still running.  0 ok, HBLS_ERR_ARG if no batch call was made yet. */
typedef struct {
    int32_t  mode;              /* 1: batched groups (+ exact pass over failed groups), 0: exact per round */
    int32_t  group_size;        /* G (4 or 8) in mode 1, else 0 */
    uint64_t rounds;            /* items in the call */
    uint64_t groups;            /* groups tested in mode 1 */
    uint32_t groups_failed;     /* groups the batched test rejected (bad or undecodable round inside) */
    uint32_t rounds_rechecked;  /* rounds the exact pass re-verified because their group failed */
    uint32_t tail_rounds;       /* rounds outside any group (rounds mod G), always verified exactly */
    uint32_t cta_threads;       /* threads per CTA of the pairing kernel (512 = lock-stepped persistent CTAs) */
} hbls_batch_info;
int hbls_last_batch_info(hbls_batch_info* out);
/* tuning knobs (tests, sweeps): "rlc_min" (rounds from which mode 1 batches in groups), "rlc_g" (0 auto / 4 / 8), "coop_max" (exact
 * checks of at most this many rounds use the warp-per-round latency kernel, 0 = never), "tpsm" (resident threads per SM of the
 * thread-per-item kernels), "tpsm_split" (lane-pair kernels), "tpsm_light", "coop_wpsm" (resident warps per SM of the warp-per-round kernels), "hm_cache" (0: H(m) cache off), "hash_coop_max" (hash-to-G2 of at most this many messages runs one warp per message), "mask_sort" (1: large batches aggregate keys in the order of the rounds' addition counts), "hash_split" (large batches hash in 0: one kernel, 1: map + cofactor clearing, 2: map + cofactor clearing + affine conversion), "rlc_two_phase" (batched pairing as 0: one kernel, 1: two kernels when the batch fills the chip, 2: always two kernels), "hash_fallback" (test hook: 1 forces the warp-per-message hash through its complete-formula fall-back), "tpsm_sw" (resident threads per SM of the map kernel), "overlap" (1: small batches decode signatures and
 * hash messages on two auxiliary streams beside the key aggregation), "scale_split" (batched groups scale keys and signatures in 0: one
 * kernel, 1: a G1 kernel and a G2 kernel), "decode_split" (large batches decode signatures in 0: one kernel with the subgroup test,
 * 1: decode + a separate subgroup kernel), "exact_two_phase" (1: exact checks beyond coop_max and the exact pass over failed groups run
 * as line kernel + accumulator kernel when rlc_two_phase is 2), "tpsm_cof", "tpsm_dec", "tpsm_scale", "tpsm_scale_g1", "tpsm_lines",
 * "tpsm_accum" (resident threads per SM of the cofactor, decode, scaling, line and accumulator kernels).  Defaults come from HBLS_RLC_MIN, HBLS_RLC_G, HBLS_COOP_MAX,
 * HBLS_TPSM, HBLS_TPSM_SPLIT, HBLS_TPSM_LIGHT at blsInit.  0 ok, HBLS_ERR_ARG for an unknown name / bad value. */
int hbls_set_param(const char* name, long long value);
long long hbls_get_param(const char* name);
/* same, every pointer already in device memory (HBM); stream = cudaStream_t or NULL; asynchronous on that stream */
int hbls_aggregate_verify_batch_device(const hbls_committee* c, size_t B, const void* d_bitmaps, size_t blen,
                                       const void* d_sigs96, const void* d_msgs, size_t msg_len,
                                       void* d_results, void* stream);

/* k independent (pk, msg, sig) triples (leader onPrepare/onCommit loop consensus/leader.go:127-182,227-290;
 * view-change storm consensus/view_change_construct.go:237-375): results[j] = Deserialize ok && VerifyHash. */
int hbls_verify_batch(size_t k, const uint8_t* pk48, const uint8_t* sig96, const uint8_t* msgs, size_t msg_len,
                      uint8_t* results);
/* Same check with the reason of a failure, in the order the reference meets the errors when it parses and then checks a
 * message (consensus/view_change_msg.go:139-190 ParseViewChangeMessage: BytesToBLSPublicKey(sender), Sign.Deserialize; then
 * consensus/checks.go:20-39 verifyMessageSig / checks.go:186, view_change_construct.go:266,339 VerifyHash):
 *   HBLS_VB_BAD_KEY_ENCODING  pk48 does not decode to a point of G1 (crypto/bls/mask.go:35-55 returns the error)
 *   HBLS_VB_BAD_SIG_ENCODING  sig96 does not decode to a point of G2 ("err blsSignatureDeserialize")
 *   HBLS_VB_BAD_SIG           both decode, VerifyHash(pk, msg) is false
 *   HBLS_VB_OK                valid */
#define HBLS_VB_BAD_SIG          0
#define HBLS_VB_OK               1
#define HBLS_VB_BAD_SIG_ENCODING 3
#define HBLS_VB_BAD_KEY_ENCODING 4
int hbls_verify_batch_status(size_t k, const uint8_t* pk48, const uint8_t* sig96, const uint8_t* msgs, size_t msg_len,
                             uint8_t* status);

/* Multi-committee batch (BASELINE configs[2]: 4 shards x 250 validators, 4 distinct messages, one batched pairing; crosslinks:
 * internal/chain/engine.go:592-604, node/harmony/node_cross_link.go:69-90).  Item j = (committees[j], bitmap_j, sig_j, msg_j);
 * bitmaps = the items' bitmaps back to back, item j occupying (size(committees[j]) + 7) >> 3 bytes.  results[j] = 1/0. */
int hbls_aggregate_verify_items(size_t k, const hbls_committee* const* committees, const uint8_t* bitmaps, const uint8_t* sigs96,
                                const uint8_t* msgs, size_t msg_len, uint8_t* results);

/* Block-range header verification (SURVEY 8f.1: api/service/stagedstreamsync/sig_verify.go:23-58, internal/chain/engine.go:81-97
 * VerifyHeaders, engine.go:619-642 verifySignature) for n headers signed by ONE committee epoch, in one device call.
 * Header i: sigs96[i] = LastCommitSignature, bitmaps[i] = LastCommitBitmap (blen bytes), payloads[i] = ConstructCommitPayload(...)
 * (payload_len = 40 or 48).  quorum = minimum number of set bits among the n_committee slots (uniform vote: 2n/3 + 1,
 * consensus/quorum/one-node-one-vote.go:57-72); 0 skips the gate (staked-vote deciders apply theirs in Go).
 * status[i] follows the order of checks in engine.go:630-640:
 *   HBLS_HDR_BAD_ENCODING  signature bytes do not decode ("unable to deserialize multi-signature from payload")
 *   HBLS_HDR_NO_QUORUM     popcount(bitmap restricted to the committee slots) < quorum ("not enough signature collected")
 *   HBLS_HDR_BAD_SIG       aggSig.VerifyHash(mask.AggregatePublic, payload) is false
 *   HBLS_HDR_OK            valid */
#define HBLS_HDR_BAD_SIG      0
#define HBLS_HDR_OK           1
#define HBLS_HDR_NO_QUORUM    2
#define HBLS_HDR_BAD_ENCODING 3
int hbls_verify_headers(const hbls_committee* c, size_t n, const uint8_t* sigs96, const uint8_t* bitmaps, size_t blen,
                        const uint8_t* payloads, size_t payload_len, size_t quorum, uint8_t* status);

/* Persistent device Mask (SURVEY 8f.2; crypto/bls/mask.go:67-242; TODO(audit) at consensus/consensus_service.go:318): the
 * bitmap lives on the host, the running aggregate public key in HBM; SetMask / SetBit apply only the DELTA (Add on 0->1,
 * Sub on 1->0, mask.go:121-133,137-155) instead of rebuilding the sum.  Return 0 or HBLS_ERR_ARG (length / index). */
typedef struct hbls_mask hbls_mask;
int  hbls_mask_create(hbls_mask** out, const hbls_committee* c);
void hbls_mask_destroy(hbls_mask* m);
int  hbls_mask_set_mask(hbls_mask* m, const uint8_t* bitmap, size_t blen);
int  hbls_mask_set_bit(hbls_mask* m, size_t index, int enable);
int  hbls_mask_clear(hbls_mask* m);
int  hbls_mask_count_enabled(const hbls_mask* m);
/* bitmap_out (nullable, blen bytes) = Mask.Bitmap ; pk48_out (nullable) = AggregatePublic.Serialize() */
int  hbls_mask_get(const hbls_mask* m, uint8_t* bitmap_out, size_t blen, uint8_t pk48_out[48]);
/* aggSig.VerifyHash(mask.AggregatePublic, msg) with the resident aggregate (consensus/validator.go:228): 1 / 0 / <0 */
int  hbls_mask_verify(const hbls_mask* m, const uint8_t sig96[96], const void* msg, size_t msg_len);

/* Running vote aggregate (SURVEY 8f.2; consensus/quorum/quorum.go:164-196 AggregateVotes re-deserialises every stored hex
 * signature at ~0.5 ms each): votes are decoded ONCE when they arrive and folded into a device-resident G2 sum.
 * add_vote: signer_bitmap marks the vote's signer key(s) (multi-key votes set several bits, leader.go:283).  Returns 0 added,
 * 1 skipped because a signer is already collected (the de-dup rule of quorum.go:168-181), HBLS_ERR_DECODE for a bad signature. */
typedef struct hbls_ballot_box hbls_ballot_box;
int  hbls_ballot_box_create(hbls_ballot_box** out, const hbls_committee* c);
void hbls_ballot_box_destroy(hbls_ballot_box* b);
int  hbls_ballot_box_add_vote(hbls_ballot_box* b, const uint8_t* signer_bitmap, size_t blen, const uint8_t sig96[96]);
/* aggregate signature of the collected votes + their bitmap (construct.go:158-175 constructQuorumSigAndBitmap) */
int  hbls_ballot_box_aggregate(const hbls_ballot_box* b, uint8_t out_sig96[96], uint8_t* bitmap_out, size_t blen);

/* ONE batch split over several GPUs (SURVEY 8e; BASELINE configs[3] "sharded across 8 x B200 with NCCL G1/G2 partial-sum allreduce").
 * Rank g turns its slice of independent (pk, msg, sig) triples into a fixed-size partial record
 *     { sum_j r_j sigma_j (G2 Jacobian, 288 B) ; prod_j Miller(-r_j pk_j, H(m_j)) (Fp12, 576 B, no final exponentiation) ; item / bad counts }
 * with one fresh 64-bit coefficient per item; the ranks all-gather the records (EC addition and Fp12 multiplication are not NCCL
 * reduction operators, so the "allreduce" is an all-gather + identical local fold: harmony_b200/shard.py) and hbls_rlc_fold
 * multiplies the partial products, adds Miller(B, sum of the partial sums) and runs ONE final exponentiation.
 * fold returns 1 = every item of every slice is valid (error probability <= 2^-63), 0 = not proven (some item is invalid or did not
 * decode: every rank then verifies its own slice exactly with hbls_verify_batch), < 0 error. */
#define HBLS_PARTIAL_BYTES 872
int hbls_rlc_partial(size_t k, const uint8_t* pk48, const uint8_t* sig96, const uint8_t* msgs, size_t msg_len, uint8_t record[HBLS_PARTIAL_BYTES]);
int hbls_rlc_fold(size_t n_records, const uint8_t* records);

/* batched SignHash / GetPublicKey (consensus/construct.go:97-114 with multibls keys) ; ok[j] = 1/0 */
int hbls_sign_hash_batch(size_t k, const uint8_t* sk32, const uint8_t* msgs, size_t msg_len, uint8_t* sig96_out, uint8_t* ok);
int hbls_get_public_key_batch(size_t k, const uint8_t* sk32, uint8_t* pk48_out);

/* H(m) cache.  The library keeps the hash-to-G2 points of the last 64 distinct messages on the device (LRU, keyed by the 48
 * zero-padded bytes the map reads).  blsSignHash, blsVerifyHash, hbls_aggregate_verify, hbls_mask_verify and the same-message form of
 * hbls_aggregate_verify_batch fill and consult it, so a validator that signs a block hash / commit payload (consensus/validator.go
 * prepare / commit votes) finds H(m) ready when it verifies the PREPARED / COMMITTED aggregate over the same bytes
 * (validator.go:219-236) -- the reference's analogue is its LRU of decoded public keys (crypto/bls/mask.go:35-55).
 * hbls_hash_prefetch enqueues H(msg) on an auxiliary stream and returns at once (e.g. on ANNOUNCE, when block hash, number and view
 * id -- hence the commit payload -- become known).  hbls_set_param("hm_cache", 0) turns the cache off.  0 ok. */
int hbls_hash_prefetch(const void* msg, size_t msg_len);
int hbls_hash_cache_stats(uint64_t* hits, uint64_t* misses);
/* coalescing of the per-call operations (Threading above), counted since load: requests queued, batches run, largest batch.
 * requests == batches when every call ran alone.  Any pointer may be NULL.  0 ok. */
int hbls_coalesce_stats(uint64_t* requests, uint64_t* batches, uint64_t* largest_batch);

/* ------------------------------------------------------------------ probes used by tests / bench */
/* message -> G2 point, serialized (the H(m) of SignHash/VerifyHash): 0 ok, -1 undefined */
int hbls_map_to_g2(const void* msg, size_t msg_len, uint8_t out96[96]);
/* n field products on canonical little-endian 48-byte operands (kernel parity probe) */
int hbls_fp_mul_batch(size_t n, const uint8_t* a48, const uint8_t* b48, uint8_t* out48);
/* number of kernels this library has launched so far */
uint64_t hbls_kernel_launch_count(void);
/* compile-time variant of the device code: bit 0 = shared inversions (Montgomery's trick over the items of a persistent thread in
 * hash-to-G2 and coefficient scaling), bits 8.. = items per shared inversion */
int hbls_build_info(void);
/* device self-test of the lane-pair (split Fp2) primitives used by k_pairing_verify_split against the single-thread
 * primitives on pseudo-random operands: returns the number of mismatches (0 = pass), <0 on error */
int hbls_selftest_split(uint32_t iters);
/* per-kernel device timing of the aggregate-verify pipeline (CUDA events on the launching stream).
 * enable(1) makes every following hbls_aggregate_verify_batch[_device] call record events between its kernels;
 * get() waits for the last recorded pipeline and returns the number of stages written to ms_out, in launch order:
 * 0 mask aggregation, 1 (-apk to affine; exact mode only), 2 k_g2_decode, 3 k_hash_to_g2, 4 k_rlc_scale + k_rlc_group_sum, 5 pairing
 * (batched groups + exact pass over failed groups; in exact mode stage 4 is empty) */
void hbls_stage_timing_enable(int on);
int hbls_stage_timing_get(float* ms_out, int max_stages);
/* integer-pipe probe: every thread of a chip-filling grid runs `iters` rounds of the field multiplier's own carry-chained
 * mad.lo.cc / madc.hi.cc rows (IMAD.WIDE.U32.X, 4 independent accumulator sets) and the call returns the achieved 32x32+64
 * MACs per second; *sm_clock_hz (nullable) receives the device's maximum SM clock (cudaDevAttrClockRate).
 * Roofline denominator: an IMAD.WIDE holds the FMA-heavy pipe for 4 cycles per warp (profiles/r2_probe_int.*), so the
 * pipe peak is sm_count * 4 schedulers * 8 MAC/clk * SM clock (bench.py uses the clock nvidia-smi reports under load);
 * the probe itself reaches about 90 % of it.  <0 on error */
double hbls_probe_mac32_per_s(int iters, double* sm_clock_hz);

#ifdef __cplusplus
}
#endif
#endif
