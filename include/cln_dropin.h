/*
 * cln_dropin.h — the reference's own entry points for the verification path, re-implemented on top
 * of the batch engine (cln_sigverify.h).  Same names, argument meaning and error behaviour as CLN:
 *
 *   check_signed_hash          bitcoin/signature.h:85    (bitcoin/signature.c:174-192)
 *   check_signed_hash_nodeid   common/node_id.h:80       (common/node_id.c:72-80)
 *   check_schnorr_sig          bitcoin/signature.h:129   (bitcoin/signature.c:408-430)
 *   sha256_double              bitcoin/shadouble.h       (bitcoin/shadouble.c:7-11)
 *   pubkey_from_der            bitcoin/pubkey.h          (bitcoin/pubkey.c:14-24)
 *   sigcheck_channel_announcement / _node_announcement / _channel_update
 *                              gossipd/sigcheck.h        (gossipd/sigcheck.c:45-115, 118-164, 9-43)
 *                              — here in BATCH form: n raw wire messages in, one status per message out
 *   check_tx_sigs_batch        the per-HTLC loop of channeld/channeld.c:2215-2232 (one shared key,
 *                              n sighashes, n signatures) as one launch
 *
 *   check_tx_sig               bitcoin/signature.h:120   (bitcoin/signature.c:194-221) — same signature; the BIP143
 *                              sighash (bitcoin_tx_hash_for_sig :120-151 -> libwally tx_io.c:660-765) is computed
 *                              on the device from the wally_tx fields
 *
 * A false return always means "signature invalid" (peer's fault).  Engine failures (no GPU, CUDA
 * error) abort() with a message on stderr, CLN's convention for internal errors
 * (bitcoin/signature.c:117,212,420; SURVEY.md §8b) — they are never reported as false.
 *
 * Types: inside CLN the real headers provide these (define CLN_TYPES_PROVIDED before including);
 * stand-alone, layout-compatible minimal definitions are supplied below.
 */
#ifndef CLN_DROPIN_H
#define CLN_DROPIN_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef CLN_TYPES_PROVIDED
typedef unsigned char u8;
struct sha256 { union { uint32_t u32[8]; unsigned char u8[32]; } u; };  /* ccan/crypto/sha256/sha256.h */
struct sha256_double { struct sha256 sha; };                           /* bitcoin/shadouble.h:9-11 */
typedef struct { unsigned char data[64]; } secp256k1_ecdsa_signature;   /* secp256k1.h (opaque) */
typedef struct { unsigned char data[64]; } secp256k1_pubkey;            /* secp256k1.h (opaque) */
typedef struct { unsigned char data[65]; } secp256k1_ecdsa_recoverable_signature; /* secp256k1_recovery.h (opaque):
                                                   r, s as 4x64-bit little-endian limbs, recid at data[64] */
struct pubkey { secp256k1_pubkey pubkey; };                            /* bitcoin/pubkey.h:15-18 */
struct node_id { u8 k[33]; };                                          /* common/node_id.h:11-13 */
struct bip340sig { u8 u8[64]; };                                       /* bitcoin/signature.h:145-147 */
enum sighash_type { SIGHASH_ALL = 1, SIGHASH_NONE = 2, SIGHASH_SINGLE = 3, SIGHASH_ANYONECANPAY = 0x80 };
struct bitcoin_signature { secp256k1_ecdsa_signature s; enum sighash_type sighash_type; }; /* signature.h:47-50 */
/* libwally's public transaction structs (external/libwally-core/include/wally_transaction.h:89-155), Elements fields
 * included as CLN builds libwally (no WALLY_ABI_NO_ELEMENTS); only the fields BIP143 commits to are read. */
struct wally_tx_witness_stack;
struct wally_tx_input {
    unsigned char txhash[32];
    uint32_t index;
    uint32_t sequence;
    unsigned char *script;
    size_t script_len;
    struct wally_tx_witness_stack *witness;
    uint8_t features;
    unsigned char blinding_nonce[32];
    unsigned char entropy[32];
    unsigned char *issuance_amount;
    size_t issuance_amount_len;
    unsigned char *inflation_keys;
    size_t inflation_keys_len;
    unsigned char *issuance_amount_rangeproof;
    size_t issuance_amount_rangeproof_len;
    unsigned char *inflation_keys_rangeproof;
    size_t inflation_keys_rangeproof_len;
    struct wally_tx_witness_stack *pegin_witness;
};
struct wally_tx_output {
    uint64_t satoshi;
    unsigned char *script;
    size_t script_len;
    uint8_t features;
    unsigned char *asset;
    size_t asset_len;
    unsigned char *value;
    size_t value_len;
    unsigned char *nonce;
    size_t nonce_len;
    unsigned char *surjectionproof;
    size_t surjectionproof_len;
    unsigned char *rangeproof;
    size_t rangeproof_len;
};
struct wally_tx {
    uint32_t version;
    uint32_t locktime;
    struct wally_tx_input *inputs;
    size_t num_inputs;
    size_t inputs_allocation_len;
    struct wally_tx_output *outputs;
    size_t num_outputs;
    size_t outputs_allocation_len;
};
struct chainparams;
struct wally_psbt;
struct bitcoin_tx { struct wally_tx *wtx; const struct chainparams *chainparams; struct wally_psbt *psbt; }; /* bitcoin/tx.h:32-40 */
#endif

/* Optional: choose the CUDA device (default: $CLN_SIGVERIFY_DEVICE or 0).  The context is created
 * lazily on first use; one per process, as CLN's global secp256k1_ctx (common/utils.c:16). */
void cln_sigverify_init(int device);
void cln_sigverify_shutdown(void);

bool check_signed_hash(const struct sha256_double *hash, const secp256k1_ecdsa_signature *signature,
                       const struct pubkey *key);
bool check_signed_hash_nodeid(const struct sha256_double *hash, const secp256k1_ecdsa_signature *signature,
                              const struct node_id *id);
bool check_schnorr_sig(const struct sha256 *hash, const secp256k1_pubkey *pubkey, const struct bip340sig *sig);
void sha256_double(struct sha256_double *shadouble, const void *p, size_t len);
bool pubkey_from_der(const u8 *der, size_t len, struct pubkey *key);

/* bitcoin/signature.h:120.  Exactly one of redeemscript / witness_script is used (witness_script when non-NULL), both
 * are tal arrays in CLN: their length comes from tal_bytelen(), the input amount from psbt_input_get_amount(tx->psbt, in)
 * (bitcoin/signature.c:130).  Those two are CLN-internal functions: when this object is linked into a CLN daemon they are
 * picked up directly (weak references); a stand-alone user supplies them with cln_sigverify_set_tx_hooks(). */
bool check_tx_sig(const struct bitcoin_tx *tx, size_t input_num, const u8 *redeemscript, const u8 *witness_script,
                  const struct pubkey *key, const struct bitcoin_signature *sig);
void cln_sigverify_set_tx_hooks(size_t (*script_bytelen)(const void *tal_script),
                                uint64_t (*input_amount_sat)(const struct bitcoin_tx *tx, size_t input_num));

/* Public-key recovery, batched: ok[i] = secp256k1_ecdsa_recover(secp256k1_ctx, &keys[i].pubkey, &sigs[i], hashes[i].u.u8),
 * as common/bolt11.c:1043 (invoice without an `n` field) and lightningd/signmessage.c:193 (checkmessage) call it on the
 * struct secp256k1_ecdsa_recoverable_signature_parse_compact filled.  keys[i] is all zero where ok[i] is false. */
void ecdsa_recover_batch(const secp256k1_ecdsa_recoverable_signature *sigs, const struct sha256 *hashes, size_t n,
                         struct pubkey *keys, bool *ok);

/* channeld HTLC loop: ok[i] = check_signed_hash(&hashes[i], &sigs[i].s, key) for one shared key. */
void check_tx_sigs_batch(const struct sha256_double *hashes, const struct bitcoin_signature *sigs,
                         const struct pubkey *key, size_t n, bool *ok);

/* The same loop with the BIP143 sighash ALSO computed on the device (row N2): check_tx_sig (bitcoin/signature.c:194-221)
 * for n one-input one-output transactions described by sv_tx records (cln_sigverify.h); the sighash type of each
 * signature is taken from sigs[i].sighash_type and gated exactly as check_tx_sig does (:206-211: only SIGHASH_ALL or
 * SIGHASH_SINGLE|SIGHASH_ANYONECANPAY, else false). */
struct sv_tx_fields; /* = sv_tx of cln_sigverify.h */
void check_tx_sigs_bip143_batch(const void *sv_tx_array, const u8 *scripts, size_t scripts_len,
                                const struct pubkey *key, const struct bitcoin_signature *sigs, size_t n, bool *ok);

/* gossipd: status[i] = 0 if every signature of message i verifies, else 1 + the index of the FIRST bad
 * signature in the reference's checking order (channel_announcement: node_signature_1, node_signature_2,
 * bitcoin_signature_1, bitcoin_signature_2 -> 1..4; node_announcement / channel_update: 1); -1 if the
 * message is too short / malformed to locate its fields.  msgs[i] is the complete wire message
 * (2-byte type included), lens[i] its length. */
void sigcheck_channel_announcement_batch(const u8 *const *msgs, const size_t *lens, size_t n, int *status);
void sigcheck_node_announcement_batch(const u8 *const *msgs, const size_t *lens, size_t n, int *status);
/* channel_update is signed by the node found in the gossmap: the caller supplies it. */
void sigcheck_channel_update_batch(const u8 *const *msgs, const size_t *lens, const struct node_id *signers,
                                   size_t n, int *status);

#ifdef __cplusplus
}
#endif
#endif
