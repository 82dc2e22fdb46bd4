/*
 * cln_sigverify.h — C ABI of the B200 batched secp256k1 verification engine (libcln_sigverify.so).
 *
 * This is the drop-in boundary behind Core Lightning's bitcoin/signature.h surface.  Plain C,
 * plain pointers and sizes; no CUDA, torch or libsecp256k1 types appear in any signature.
 *
 * Reference interfaces each entry point replaces (paths relative to the CLN tree):
 *
 *   sv_verify_host(SV_KIND_ECDSA_XY, ...)   check_signed_hash()          bitcoin/signature.c:174-192
 *                                           (hash32, secp256k1_ecdsa_signature, struct pubkey)
 *   sv_verify_host(SV_KIND_ECDSA33, ...)    check_signed_hash_nodeid()   common/node_id.c:72-80
 *                                           (33-byte node_id decompressed per call, then as above)
 *   sv_verify_host(SV_KIND_SCHNORR, ...)    check_schnorr_sig()          bitcoin/signature.c:408-430
 *   sv_verify_host_raw(...)                 sha256_double() + the above  bitcoin/shadouble.c:7-11,
 *                                           as used by gossipd/sigcheck.c:9-43, 45-115, 118-164 and,
 *                                           with a BIP143 preimage as the span, check_tx_sig()
 *                                           bitcoin/signature.c:194-221 (the per-HTLC loop of
 *                                           channeld/channeld.c:2215-2232)
 *   sv_sha256d_host(...)                    sha256_double()              bitcoin/shadouble.c:7-11
 *   sv_pubkey_parse_host(...)               pubkey_from_der()            bitcoin/pubkey.c:14-24
 *   sv_recover_host(...)                    secp256k1_ecdsa_recover()    common/bolt11.c:1018-1050,
 *                                           lightningd/signmessage.c:178-193 (recoverable signatures)
 *   sv_enqueue_* / sv_flush                 the deferral queue a batching caller (gossipd ingest,
 *                                           SURVEY.md §8f N1) sits on; synchronous check_* = enqueue 1 + flush
 *   sv_verify_device(...)                   same kernels on device-resident arrays (bench / multi-GPU)
 *
 * Verdict semantics are those of the reference, bit for bit, INCLUDING the parse-time rejects CLN
 * performs before check_signed_hash (r >= n, s >= n: wire/fromwire.c:188-199; bad pubkey:
 * bitcoin/pubkey.c:102-113): a verdict byte is 1 iff libsecp256k1 would parse the key, parse the
 * signature and return 1 from secp256k1_ecdsa_verify / secp256k1_schnorrsig_verify.
 *
 * Error convention (SURVEY.md §8b): a verification failure is verdict 0, never an error code.
 * Engine failures (no device, CUDA error, out of memory) return a negative sv_status and leave the
 * verdict buffer untouched; there is NO CPU fallback.  The check_* drop-in wrappers in
 * cln_dropin.h abort() on engine failure, matching CLN's "internal error is fatal" style.
 *
 * Threading: one sv_ctx per thread/process (CLN daemons are single-threaded event loops).  Calls on one context
 * share its device scratch (work records, per-thread tables): issue them one at a time, on one stream at a time.
 */
#ifndef CLN_SIGVERIFY_H
#define CLN_SIGVERIFY_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sv_ctx sv_ctx;

/* item kinds (layout of the key array; msg is always 32 bytes, sig always 64 bytes) */
#define SV_KIND_ECDSA33 0  /* key = 33-byte SEC1 compressed (02/03 || x)           sig = r_be32 || s_be32 */
#define SV_KIND_ECDSA_XY 1 /* key = 64 bytes x_be32 || y_be32 (pre-decompressed)   sig = r_be32 || s_be32 */
#define SV_KIND_SCHNORR 2  /* key = 32-byte x-only (BIP-340)                        sig = R.x_be32 || s_be32 */

typedef enum {
    SV_OK = 0,
    SV_ERR_NO_DEVICE = -1,
    SV_ERR_CUDA = -2,
    SV_ERR_NOMEM = -3,
    SV_ERR_ARG = -4
} sv_status;

/* Create an engine on CUDA device `device` (ordinal).  Allocates the stream, builds the 34 MiB
 * fixed-base table on the device (kernel K4) and the per-thread scratch.  */
int sv_create(sv_ctx **out, int device);
void sv_destroy(sv_ctx *ctx);
/* last error text for this context (or for a failed sv_create when ctx == NULL) */
const char *sv_last_error(const sv_ctx *ctx);
/* size of the key element for a kind (33 / 64 / 32), or 0 */
size_t sv_key_size(int kind);

/* ---- synchronous batch verification, HOST buffers (SoA): msg32[n][32], key[n][keysize], sig64[n][64];
 *      verdicts[n] receives 0/1.  Copies in, runs the kernels, copies out, returns when done. ---- */
int sv_verify_host(sv_ctx *ctx, int kind, const uint8_t *msg32, const uint8_t *key, const uint8_t *sig64,
                   size_t n, uint8_t *verdicts);

/* Batches of at most `small_max` signatures (default = capacity = 8192; 0 disables) take the LATENCY path: one launch
 * of a kernel that spreads each verification over three warps (key side / scalar side in parallel, then the two GLV
 * half-ladders and the fixed-base comb in parallel, joined by full Jacobian additions), inputs and verdicts passing
 * through a pinned, device-mapped staging block (no copy commands, no allocation).  Larger batches take the throughput
 * kernels.  Verdicts are identical on both paths (tests/test_gpu_small.py). */
int sv_set_small_max(sv_ctx *ctx, size_t small_max);
size_t sv_get_small_max(const sv_ctx *ctx);

/* ---- MIXED batch (BASELINE config C3: interleaved ECDSA + BIP-340): kinds[i] is the SV_KIND_* tag of item i, keys sit
 *      in 64-byte slots (the first 33 / 64 / 32 bytes are the key).  The batch is split per kind on the device (index
 *      lists by warp-aggregated atomics, gather, per-kind kernels, scatter); verdicts come back in item order; an
 *      unknown tag yields verdict 0. ---- */
int sv_verify_mixed_host(sv_ctx *ctx, const uint8_t *kinds, const uint8_t *msg32, const uint8_t *key64,
                         const uint8_t *sig64, size_t n, uint8_t *verdicts);
int sv_verify_mixed_device(sv_ctx *ctx, const void *d_kinds, const void *d_msg32, const void *d_key64,
                           const void *d_sig64, size_t n, void *d_verdicts, void *stream);

/* ---- same, but the message hash is computed on the device: item i signs
 *      SHA256d(data[off[i] .. off[i]+len[i])).  Several items may share one span (the four
 *      signatures of a channel_announcement do). ---- */
int sv_verify_host_raw(sv_ctx *ctx, int kind, const uint8_t *data, size_t data_len, const uint64_t *off,
                       const uint32_t *len, const uint8_t *key, const uint8_t *sig64, size_t n,
                       uint8_t *verdicts);

/* ---- gossip ingest with DEVICE-side slicing (SURVEY.md §8f N1; replaces the per-message work of
 *      gossipd/sigcheck.c:9-164 and the field extraction of wire/peer_wiregen.c for the three gossip messages):
 *      blob = concatenated raw wire messages (2-byte type included), msg_off/msg_len locate them.  The device finds
 *      the signatures, keys and signed regions itself, hashes (SHA-256d) and verifies.  status[m] = 0 all signatures
 *      good; 1..4 = first bad signature in the reference's order (node_signature_1, node_signature_2,
 *      bitcoin_signature_1, bitcoin_signature_2; node_announcement / channel_update: 1); -1 = not a gossip message,
 *      shorter than the message's fixed layout (every field of wire/peer_wire.csv:340-377 up to and including the
 *      variable-length features / addresses arrays must be present, as the generated fromwire_* require), a signature
 *      with r or s >= n, or an undecodable bitcoin_key.  NOT checked: the TLV stream that may follow a
 *      node_announcement (node_ann_tlvs) — a caller that consumes those still parses them itself.  channel_update is signed by a node the caller looks up in its gossmap: cu_signers33[m] (33 bytes per
 *      MESSAGE, ignored for other types; NULL if the batch has no channel_update). ---- */
int sv_verify_gossip_host(sv_ctx *ctx, const uint8_t *blob, size_t blob_len, const uint64_t *msg_off,
                          const uint32_t *msg_len, size_t n_msgs, const uint8_t *cu_signers33, int *status);

/* L2 residency hint for the throughput kernels (default on): the G comb table and the per-thread multiples tables are
 * marked persisting through a stream access-policy window, the rest of the stream's traffic streaming.  0 switches it off
 * for streams not yet seen (measurement aid). */
int sv_set_l2_policy(sv_ctx *ctx, int on);

/* ---- BIP-340 BATCH verification by random linear combination (SURVEY.md 8f N3; BIP-340 "Batch Verification").  The batch
 *      is cut into groups of 1024 signatures; each group's equation  sum a_i R_i + sum a_i e_i P_i - (sum a_i s_i) G = 0
 *      is evaluated with a per-warp bucket method (about half the field work of one-by-one verification); the members of
 *      a group whose equation fails are re-verified one by one, so every verdict is the one sv_verify_host(SV_KIND_SCHNORR)
 *      gives, up to the 2^-127 chance that random a_i hide a bad signature.  Meant for batches that are almost all valid
 *      (a bad signature costs its whole group the fast path).  seed32: 32 bytes the signers could not predict (NULL: taken
 *      from getrandom()).  groups_total / groups_failed (optional) report how the batch went. ---- */
int sv_verify_schnorr_batch_host(sv_ctx *ctx, const uint8_t *msg32, const uint8_t *xonly32, const uint8_t *sig64, size_t n,
                                 const uint8_t *seed32, uint8_t *verdicts, uint32_t *groups_total, uint32_t *groups_failed);

/* Key de-duplication (SURVEY.md 8f N3): sv_verify_gossip_host looks for repeated keys in batches above the small-batch limit (and >= 4096 signatures)
 * (exact hash table over the 33 key bytes, on the device); when at least 40 % of the items repeat a key, every DISTINCT
 * key is decoded and its multiples table built once and the curve kernel indexes those tables.  Verdicts are unchanged.
 * sv_set_dedup(ctx, 0) switches the search off; sv_last_distinct_keys reports what the last gossip batch contained. */
int sv_set_dedup(sv_ctx *ctx, int on);
unsigned sv_last_distinct_keys(const sv_ctx *ctx);

/* Compressed-key ECDSA (SV_KIND_ECDSA33) batches above the small-batch limit never take the square root of
 * secp256k1_eckey_pubkey_parse (eckey_impl.h:17-20 -> group_impl.h:334-346): the unknown y only scales Z, the final
 * comparison becomes linear in y and is settled by one batched division (lightning_b200/csrc/verify.cuh, "without the
 * square root").  Verdicts are identical; sv_set_nosqrt(ctx, 0) selects the plain flow (A/B measurements, tests). */
int sv_set_nosqrt(sv_ctx *ctx, int on);

/* ---- n ECDSA signatures by ONE key (SURVEY.md §8a a16 / §8f N3: every HTLC signature of a commitment_signed is made
 *      with remote_htlckey, channeld/channeld.c:2154,2215-2232).  The key is decoded and its multiples table built once;
 *      each verification skips the per-signature square root and table build.  kind: SV_KIND_ECDSA33 or _XY; key is
 *      ONE key of that kind. ---- */
int sv_verify_samekey_host(sv_ctx *ctx, int kind, const uint8_t *key, const uint8_t *msg32, const uint8_t *sig64,
                           size_t n, uint8_t *verdicts);

/* ---- check_tx_sig with the BIP143 sighash computed ON THE DEVICE (SURVEY.md §8f N2).  Replaces, for the one-input
 *      one-output commitment-HTLC transactions of channeld/channeld.c:2215-2232 (shape: common/htlc_tx.c:10-69),
 *      bitcoin_tx_hash_for_sig (bitcoin/signature.c:120-151) -> wally_tx_get_btc_signature_hash ->
 *      bip143_signature_hash (libwally tx_io.c:660-765) + check_signed_hash.  The host passes only the fields of the
 *      preimage; scripts live in one blob.  Multi-output / multi-input transactions (the commitment transaction itself,
 *      check_tx_sig in general) pass their serialised outputs / outpoints through the SV_TX_* flags.  sighash32_out (optional, n x 32) returns the computed sighashes. ---- */
#define SV_TX_OUTPUTS_SERIALIZED 1u /* the out_script span holds the already-serialised outputs to commit to (amount ||
                                       CompactSize || script, concatenated: all outputs for SIGHASH_ALL, the one at the
                                       input's index for SIGHASH_SINGLE); output_amount is ignored */
#define SV_TX_INPUTS_SERIALIZED 2u  /* multi-input transaction: the prevouts span holds every outpoint (36 bytes each), the
                                       sequences span every nSequence (4 bytes each) — hashPrevouts / hashSequence are
                                       taken over them; prev_txid/prev_index/sequence still describe THE input being signed */
#define SV_TX_OUTPUTS_ZERO 4u       /* hashOutputs is 32 zero bytes (SIGHASH_SINGLE with no output at the input's index,
                                       libwally tx_io.c:725) */
typedef struct {
    uint32_t version, locktime, sequence, sighash_type; /* sighash_type: SIGHASH_ALL 1 / NONE 2 / SINGLE 3, | 0x80 ANYONECANPAY */
    uint8_t prev_txid[32];                              /* as serialised in the transaction (internal byte order) */
    uint32_t prev_index;
    uint32_t script_off, script_len;                    /* witness script (scriptCode) inside `scripts`, any length */
    uint32_t out_script_off, out_script_len;            /* scriptPubKey of the single output inside `scripts` (or the
                                                           serialised outputs, see SV_TX_OUTPUTS_SERIALIZED) */
    uint32_t flags;                                     /* 0 for the one-input one-output HTLC shape, or SV_TX_* above */
    uint64_t input_amount, output_amount;               /* satoshi */
    uint32_t prevouts_off, prevouts_len;                /* SV_TX_INPUTS_SERIALIZED only */
    uint32_t sequences_off, sequences_len;
} sv_tx;
int sv_verify_tx_host(sv_ctx *ctx, int kind, const sv_tx *txs, const uint8_t *scripts, size_t scripts_len,
                      const uint8_t *key, const uint8_t *sig64, size_t n, uint8_t *verdicts, uint8_t *sighash32_out);

/* ---- ECDSA PUBLIC-KEY RECOVERY, batched: secp256k1_ecdsa_recoverable_signature_parse_compact + secp256k1_ecdsa_recover
 *      (modules/recovery/main_impl.h:38-57, 137-156) as common/bolt11.c:1018-1050 (invoice signatures without an `n`
 *      field) and lightningd/signmessage.c:178-193 (checkmessage) call them.  Inputs: msg32[n][32], sig64[n][64] = r_be32 ||
 *      s_be32 (compact form), recid[n] one byte each.  Outputs per item:
 *        status[i] = -1  encoding refused: r >= n, s >= n or recid > 3 (never an abort);
 *        status[i] =  0  no key: r == 0, s == 0, recid & 2 with r >= p - n, x = r (+ n) not on the curve, or Q = infinity;
 *                        xy64[i] is all zero (as the reference clears its output);
 *        status[i] =  1  xy64[i] = x_be32 || y_be32 of Q = (-m/r)*G + (s/r)*R, the form sv_pubkey_parse_host writes.
 *      m = msg mod n is never rejected, and there is no low-S rule: a high s recovers.  Batches of at most small_max items
 *      take the small-batch kernel, larger ones the throughput kernels in SV_HOST_CHUNK slices; sv_set_profiling events
 *      cover the scalar-side and curve-side kernels.  Not available in mixed batches or the deferral queue. ---- */
int sv_recover_host(sv_ctx *ctx, const uint8_t *msg32, const uint8_t *sig64, const uint8_t *recid, size_t n,
                    uint8_t *xy64, int8_t *status);

/* ---- DEVICE buffers (same SoA layout, device pointers); asynchronous on `stream`
 *      (a cudaStream_t passed as void*; NULL = the context's own stream).  d_verdicts[n] bytes;
 *      d_bitmap, if non-NULL, receives ceil(n/32) little-endian 32-bit words, bit i%32 of word i/32. ---- */
int sv_verify_device(sv_ctx *ctx, int kind, const void *d_msg32, const void *d_key, const void *d_sig64, size_t n,
                     void *d_verdicts, void *d_bitmap, void *stream);
int sv_sync(sv_ctx *ctx, void *stream);
/* the context's own cudaStream_t (as void*), e.g. to record timing events on it */
void *sv_get_stream(const sv_ctx *ctx);

/* ---- deferral queue: enqueue returns the item's index in the pending batch; sv_flush verifies all
 *      pending items of every kind and writes one verdict byte per item in enqueue order. ---- */
long sv_enqueue(sv_ctx *ctx, int kind, const uint8_t msg32[32], const uint8_t *key, const uint8_t sig64[64]);
size_t sv_pending(const sv_ctx *ctx);
int sv_flush(sv_ctx *ctx, uint8_t *verdicts, size_t capacity);

/* ---- helpers of the bitcoin/ surface that are pure functions of bytes ---- */
/* out32[i] = SHA256d(data[off[i]..off[i]+len[i]))   (bitcoin/shadouble.c:7) */
int sv_sha256d_host(sv_ctx *ctx, const uint8_t *data, size_t data_len, const uint64_t *off, const uint32_t *len,
                    size_t n, uint8_t *out32);
/* pubkey_from_der semantics for a batch: key33[n][33] -> xy64[n][64] (x||y big-endian), ok[n] = 0/1 */
int sv_pubkey_parse_host(sv_ctx *ctx, const uint8_t *key33, size_t n, uint8_t *xy64, uint8_t *ok);

/* ---- device-side self test of the arithmetic (TEST SUPPORT; model: libsecp256k1 tests.c:3023-3176 field self-tests,
 *      :2354 scalar tests).  Runs ONE primitive of the engine's inline-PTX arithmetic on caller operands, one GPU thread
 *      per item: a[n][8], b[n][8] little-endian 32-bit limbs in; out[n][16] limbs out (result in out[0..7]; flags or the
 *      high half in out[8..15], see the list).  Field results are in the engine's WEAK form (any value < 2^256
 *      congruent to the residue) unless stated. ---- */
enum {
    SV_ST_FE_MUL = 0,        /* a*b mod p */
    SV_ST_FE_SQR = 1,        /* a^2 */
    SV_ST_FE_ADD = 2,        /* a+b */
    SV_ST_FE_SUB = 3,        /* a-b */
    SV_ST_FE_NEG = 4,        /* -a */
    SV_ST_FE_NORMALIZE = 5,  /* canonical a; out[8] = (a == 0 mod p), out[9] = (a >= p), out[10] = (a == b mod p) */
    SV_ST_FE_INV = 6,        /* a^(p-2) */
    SV_ST_FE_SQRT = 7,       /* a^((p+1)/4); out[8] = 1 iff it squares back to a */
    SV_ST_FE_MUL3 = 8,
    SV_ST_FE_MUL8 = 9,
    SV_ST_FE_MUL_SMALL = 10, /* a * (b[0] & 0xFFFF) */
    SV_ST_FE_DBL = 11,
    SV_ST_FE_B32 = 12,       /* a = 32 big-endian bytes (memory order): set_b32 -> get_b32 round trip; out[8] = (value < p) */
    SV_ST_U256_MUL_WIDE = 13, /* full 512-bit product in out[0..15] */
    SV_ST_U256_SQR_WIDE = 14,
    SV_ST_FE_REDUCE512 = 15,  /* (a + b*2^256) mod p */
    SV_ST_U256_ADD = 16,      /* out[8] = carry */
    SV_ST_U256_SUB = 17,      /* out[8] = borrow */
    SV_ST_SC_MUL = 20,        /* a*b mod n (a, b < n), canonical */
    SV_ST_SC_SQR = 21,
    SV_ST_SC_ADD = 22,
    SV_ST_SC_NEGATE = 23,     /* out[8] = is_high(a), out[9] = is_zero(a), out[10] = (a >= n) */
    SV_ST_SC_INVERSE = 24,
    SV_ST_SC_REDUCE512 = 25,  /* (a + b*2^256) mod n */
    SV_ST_SC_SPLIT_LAMBDA = 26, /* r1 -> out[0..7], r2 -> out[8..15] */
    SV_ST_SC_SET_B32 = 27,    /* a = 32 big-endian bytes: reduced scalar, out[8] = overflow */
    SV_ST_ECMULT_GEN = 28,    /* a*G through the fixed-base comb table: affine x -> out[0..7], y -> out[8..15]; 0 -> zeros */
    SV_ST_PREPARE_U2 = 29,    /* b = u2: |k1| -> out[0..4], |k2| -> out[5..9] (sign in bit 159), both odd */
    SV_ST_PREPARE_U1 = 30,    /* a = u1: 16 signed comb digits -> out[0..15] */
    SV_ST_SC_INVERSE_VAR = 31, /* binary extended Euclid: same value as SV_ST_SC_INVERSE */
    SV_ST_FE_INV_VAR = 32     /* canonical 1/a mod p */
};
int sv_selftest_host(sv_ctx *ctx, int op, const uint32_t *a, const uint32_t *b, size_t n, uint32_t *out);

/* ---- synthetic workload generator (benchmark / test support; NOT constant time, no secrets):
 *      item i gets secret key and nonce derived from (seed, i); writes msg32, key (per kind) and a
 *      VALID low-S ECDSA / BIP-340 signature to device arrays. ---- */
int sv_synth_device(sv_ctx *ctx, int kind, uint64_t seed, size_t n, void *d_msg32, void *d_key, void *d_sig64,
                    void *stream);

/* ---- introspection for the benchmark ---- */
typedef struct {
    int device;
    int sm_count;
    int main_block;       /* threads per CTA of the curve-side kernel */
    int main_grid;        /* CTAs */
    int main_regs;        /* registers per thread (cudaFuncGetAttributes) */
    size_t gtable_bytes;
    size_t scratch_bytes;
    unsigned long long launches; /* kernels launched by this context so far */
    size_t l2_persist_bytes;     /* persisting L2 carve-out behind the table-slab access-policy window (0: hint off) */
    size_t l2_max_persist_bytes; /* what the device would allow */
} sv_info;
int sv_get_info(const sv_ctx *ctx, sv_info *info);

/* per-kernel device timing: when enabled, every sv_verify_* call records CUDA events on its launch stream
 * around the scalar-side and curve-side kernels; read them back after synchronising. */
int sv_set_profiling(sv_ctx *ctx, int on);
int sv_get_last_timing(sv_ctx *ctx, float *prep_ms, float *main_ms);

/* integer-pipe roofline probe: runs a dependent-chain IMAD.WIDE.U32 microbenchmark and returns the
 * achieved 32x32->64 multiply-accumulates per second on this device (the roofline denominator
 * SURVEY.md §8d asks to be measured, not assumed). */
int sv_probe_imad_peak(sv_ctx *ctx, double *imad_per_sec);
/* individual probes (see engine.cu k_probe_*): 0 IMAD.WIDE peak, 1 4-deep carry chains, 2 fe_mul/s, 3 fe_sqr/s,
 * 4 8-deep carry chains, 5 carry-save, 6 32-bit IMAD lo/hi, 7 IADD3 carry chains, 8 FP64 FMA,
 * 9 / 10: dependent fe_mul / fe_sqr per second of ONE thread on an otherwise idle device (small-batch latency model) */
int sv_probe(sv_ctx *ctx, int mode, double *ops_per_sec);

/* pinned host memory (cudaHostAlloc) for callers that want full-speed copies */
void *sv_host_alloc(size_t bytes);
void sv_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif
