/*
 * cln_dropin.c — host side of the drop-in (plain C, as the reference's bitcoin/signature.c is).
 * It only marshals bytes: opaque libsecp256k1 structs -> wire form, wire messages -> (span, key,
 * signature) items, and calls the batch C ABI.  No arithmetic happens on the host.
 */
#include "../../include/cln_dropin.h"
#include "../../include/cln_sigverify.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#if !defined(__BYTE_ORDER__) || __BYTE_ORDER__ != __ORDER_LITTLE_ENDIAN__
#error "opaque-struct conversion below assumes a little-endian 64-bit libsecp256k1 build"
#endif

static sv_ctx *g_ctx;
static int g_device = -1;

static void die(const char *what, int rc) {
    fprintf(stderr, "cln_sigverify: %s failed (%d): %s\n", what, rc, sv_last_error(g_ctx));
    abort(); /* internal error is fatal (CLN convention); never reported as "bad signature" */
}

static sv_ctx *ctx(void) {
    if (!g_ctx) {
        int dev = g_device;
        if (dev < 0) {
            const char *e = getenv("CLN_SIGVERIFY_DEVICE");
            dev = e ? atoi(e) : 0;
        }
        int rc = sv_create(&g_ctx, dev);
        if (rc != SV_OK) {
            fprintf(stderr, "cln_sigverify: sv_create(device %d) failed (%d): %s\n", dev, rc, sv_last_error(NULL));
            abort();
        }
    }
    return g_ctx;
}

void cln_sigverify_init(int device) {
    g_device = device;
    (void)ctx();
}
void cln_sigverify_shutdown(void) {
    if (g_ctx) sv_destroy(g_ctx);
    g_ctx = NULL;
}

/* libsecp256k1's opaque structs hold r,s / x,y as 4x64-bit little-endian limbs on 64-bit little-endian
 * builds (secp256k1.c:337-359, group_impl.h:968-986): 32 bytes little-endian each.  Inside CLN one would
 * call secp256k1_ecdsa_signature_serialize_compact / secp256k1_ec_pubkey_serialize instead
 * (INTEGRATION.md); the engine deliberately does not link libsecp256k1. */
static void rev32(u8 *out, const unsigned char *in) {
    for (int i = 0; i < 32; i++) out[i] = in[31 - i];
}
static void sig_to_wire(u8 out[64], const secp256k1_ecdsa_signature *s) {
    rev32(out, s->data);
    rev32(out + 32, s->data + 32);
}
static void pubkey_to_xy(u8 out[64], const secp256k1_pubkey *p) {
    rev32(out, p->data);
    rev32(out + 32, p->data + 32);
}

bool check_signed_hash(const struct sha256_double *hash, const secp256k1_ecdsa_signature *signature,
                       const struct pubkey *key) {
    u8 sig[64], xy[64], v = 0;
    sig_to_wire(sig, signature);
    pubkey_to_xy(xy, &key->pubkey);
    int rc = sv_verify_host(ctx(), SV_KIND_ECDSA_XY, hash->sha.u.u8, xy, sig, 1, &v);
    if (rc != SV_OK) die("sv_verify_host", rc);
    return v == 1;
}

bool check_signed_hash_nodeid(const struct sha256_double *hash, const secp256k1_ecdsa_signature *signature,
                              const struct node_id *id) {
    u8 sig[64], v = 0;
    sig_to_wire(sig, signature);
    int rc = sv_verify_host(ctx(), SV_KIND_ECDSA33, hash->sha.u.u8, id->k, sig, 1, &v);
    if (rc != SV_OK) die("sv_verify_host", rc);
    return v == 1;
}

bool check_schnorr_sig(const struct sha256 *hash, const secp256k1_pubkey *pubkey, const struct bip340sig *sig) {
    /* signature.c:412-423: serialize compressed, drop the parity byte -> x-only key */
    u8 xy[64], v = 0;
    pubkey_to_xy(xy, pubkey);
    int rc = sv_verify_host(ctx(), SV_KIND_SCHNORR, hash->u.u8, xy, sig->u8, 1, &v);
    if (rc != SV_OK) die("sv_verify_host", rc);
    return v == 1;
}

void sha256_double(struct sha256_double *shadouble, const void *p, size_t len) {
    uint64_t off = 0;
    uint32_t l = (uint32_t)len;
    u8 dummy = 0;
    int rc = sv_sha256d_host(ctx(), len ? (const u8 *)p : &dummy, len, &off, &l, 1, shadouble->sha.u.u8);
    if (rc != SV_OK) die("sv_sha256d_host", rc);
}

bool pubkey_from_der(const u8 *der, size_t len, struct pubkey *key) {
    if (len != 33) return false; /* PUBKEY_CMPR_LEN, bitcoin/pubkey.c:16 */
    u8 xy[64], ok = 0;
    int rc = sv_pubkey_parse_host(ctx(), der, 1, xy, &ok);
    if (rc != SV_OK) die("sv_pubkey_parse_host", rc);
    if (!ok) return false;
    rev32(key->pubkey.data, xy);
    rev32(key->pubkey.data + 32, xy + 32);
    return true;
}

/* ---- check_tx_sig (bitcoin/signature.c:194-221): gate on the sighash type, BIP143 sighash on the device from the
 * wally_tx fields (every output / outpoint is handed over serialised; the host hashes nothing), then the verification ---- */
struct amount_sat { uint64_t satoshis; };                                        /* common/amount.h */
extern size_t tal_bytelen(const void *ptr) __attribute__((weak));               /* ccan/tal/tal.h */
extern struct amount_sat psbt_input_get_amount(const struct wally_psbt *psbt, size_t in) __attribute__((weak)); /* bitcoin/psbt.h */
static size_t (*g_bytelen)(const void *);
static uint64_t (*g_input_sat)(const struct bitcoin_tx *, size_t);

void cln_sigverify_set_tx_hooks(size_t (*script_bytelen)(const void *), uint64_t (*input_amount_sat)(const struct bitcoin_tx *, size_t)) {
    g_bytelen = script_bytelen;
    g_input_sat = input_amount_sat;
}

static size_t put_varint(u8 *p, uint64_t v) { /* Bitcoin CompactSize */
    if (v < 0xfd) { p[0] = (u8)v; return 1; }
    if (v <= 0xffff) { p[0] = 0xfd; p[1] = (u8)v; p[2] = (u8)(v >> 8); return 3; }
    p[0] = 0xfe;
    for (int i = 0; i < 4; i++) p[1 + i] = (u8)(v >> (8 * i));
    return 5;
}
static size_t put_output(u8 *p, const struct wally_tx_output *o) {
    size_t n = 0;
    for (int i = 0; i < 8; i++) p[n++] = (u8)(o->satoshi >> (8 * i));
    n += put_varint(p + n, o->script_len);
    if (o->script_len) memcpy(p + n, o->script, o->script_len);
    return n + o->script_len;
}

bool check_tx_sig(const struct bitcoin_tx *tx, size_t input_num, const u8 *redeemscript, const u8 *witness_script,
                  const struct pubkey *key, const struct bitcoin_signature *sig) {
    const u8 *script = witness_script ? witness_script : redeemscript;
    /* "We only support a limited subset of sighash types." (signature.c:205-211) */
    if (sig->sighash_type != SIGHASH_ALL) {
        if (!witness_script) return false;
        if ((int)sig->sighash_type != (SIGHASH_SINGLE | SIGHASH_ANYONECANPAY)) return false;
    }
    const struct wally_tx *w = tx->wtx;
    if (input_num >= w->num_inputs) { /* assert(input_num < tx->wtx->num_inputs), signature.c:212 */
        fprintf(stderr, "cln_sigverify: check_tx_sig: input %zu of %zu\n", input_num, w->num_inputs);
        abort();
    }
    size_t script_len;
    uint64_t amount;
    if (g_bytelen) script_len = script ? g_bytelen(script) : 0;
    else if (tal_bytelen) script_len = script ? tal_bytelen(script) : 0;
    else die("check_tx_sig: no tal_bytelen (cln_sigverify_set_tx_hooks)", -4);
    if (g_input_sat) amount = g_input_sat(tx, input_num);
    else if (psbt_input_get_amount) amount = psbt_input_get_amount(tx->psbt, input_num).satoshis;
    else die("check_tx_sig: no psbt_input_get_amount (cln_sigverify_set_tx_hooks)", -4);

    const bool single = ((int)sig->sighash_type & 0x1f) == SIGHASH_SINGLE;
    size_t out_bytes = 0;
    for (size_t i = 0; i < w->num_outputs; i++) out_bytes += 8 + 5 + w->outputs[i].script_len;
    size_t cap = script_len + out_bytes + 40 * w->num_inputs + 16;
    u8 *blob = (u8 *)malloc(cap);
    if (!blob) die("malloc", -3);
    sv_tx t;
    memset(&t, 0, sizeof t);
    size_t n = 0;
    t.version = w->version;
    t.locktime = w->locktime;
    t.sequence = w->inputs[input_num].sequence;
    t.sighash_type = (uint32_t)sig->sighash_type;
    memcpy(t.prev_txid, w->inputs[input_num].txhash, 32);
    t.prev_index = w->inputs[input_num].index;
    t.input_amount = amount;
    t.script_off = (uint32_t)n;
    t.script_len = (uint32_t)script_len;
    if (script_len) memcpy(blob + n, script, script_len);
    n += script_len;
    t.out_script_off = (uint32_t)n;
    if (single) { /* the output at the input's index, or none (tx_io.c:725-731) */
        if (input_num < w->num_outputs) { n += put_output(blob + n, &w->outputs[input_num]); t.flags |= SV_TX_OUTPUTS_SERIALIZED; }
        else t.flags |= SV_TX_OUTPUTS_ZERO;
    } else {
        for (size_t i = 0; i < w->num_outputs; i++) n += put_output(blob + n, &w->outputs[i]);
        t.flags |= SV_TX_OUTPUTS_SERIALIZED;
    }
    t.out_script_len = (uint32_t)(n - t.out_script_off);
    if (w->num_inputs > 1) {
        t.flags |= SV_TX_INPUTS_SERIALIZED;
        t.prevouts_off = (uint32_t)n;
        for (size_t i = 0; i < w->num_inputs; i++) {
            memcpy(blob + n, w->inputs[i].txhash, 32);
            for (int b = 0; b < 4; b++) blob[n + 32 + b] = (u8)(w->inputs[i].index >> (8 * b));
            n += 36;
        }
        t.prevouts_len = (uint32_t)(n - t.prevouts_off);
        t.sequences_off = (uint32_t)n;
        for (size_t i = 0; i < w->num_inputs; i++) {
            for (int b = 0; b < 4; b++) blob[n + b] = (u8)(w->inputs[i].sequence >> (8 * b));
            n += 4;
        }
        t.sequences_len = (uint32_t)(n - t.sequences_off);
    }
    u8 xy[64], s64[64], v = 0;
    pubkey_to_xy(xy, &key->pubkey);
    sig_to_wire(s64, &sig->s);
    int rc = sv_verify_tx_host(ctx(), SV_KIND_ECDSA_XY, &t, blob, n, xy, s64, 1, &v, NULL);
    free(blob);
    if (rc != SV_OK) die("sv_verify_tx_host", rc);
    return v == 1;
}

void ecdsa_recover_batch(const secp256k1_ecdsa_recoverable_signature *sigs, const struct sha256 *hashes, size_t n,
                         struct pubkey *keys, bool *ok) {
    if (n == 0) return;
    u8 *buf = (u8 *)malloc(n * (32 + 64 + 1 + 64 + 1));
    if (!buf) die("malloc", -3);
    u8 *msg = buf, *sig = msg + 32 * n, *recid = sig + 64 * n, *xy = recid + n;
    int8_t *st = (int8_t *)(xy + 64 * n);
    for (size_t i = 0; i < n; i++) {
        memcpy(msg + 32 * i, hashes[i].u.u8, 32);
        rev32(sig + 64 * i, sigs[i].data);  /* r, s: 4x64-bit little-endian limbs (recovery/main_impl.h:12-35) */
        rev32(sig + 64 * i + 32, sigs[i].data + 32);
        recid[i] = sigs[i].data[64];
    }
    int rc = sv_recover_host(ctx(), msg, sig, recid, n, xy, st);
    if (rc != SV_OK) die("sv_recover_host", rc);
    for (size_t i = 0; i < n; i++) {
        ok[i] = st[i] == 1;
        rev32(keys[i].pubkey.data, xy + 64 * i);  /* all zero where nothing was recovered, as the reference leaves it */
        rev32(keys[i].pubkey.data + 32, xy + 64 * i + 32);
    }
    free(buf);
}

void check_tx_sigs_batch(const struct sha256_double *hashes, const struct bitcoin_signature *sigs,
                         const struct pubkey *key, size_t n, bool *ok) {
    if (n == 0) return;
    u8 *buf = (u8 *)malloc(n * (32 + 64 + 1));
    if (!buf) die("malloc", -3);
    u8 xy[64];
    u8 *msg = buf, *sig = buf + 32 * n, *v = sig + 64 * n;
    pubkey_to_xy(xy, &key->pubkey);
    for (size_t i = 0; i < n; i++) {
        memcpy(msg + 32 * i, hashes[i].sha.u.u8, 32);
        sig_to_wire(sig + 64 * i, &sigs[i].s);
    }
    /* one key for the whole loop: its multiples table is built once on the device */
    int rc = sv_verify_samekey_host(ctx(), SV_KIND_ECDSA_XY, xy, msg, sig, n, v);
    if (rc != SV_OK) die("sv_verify_samekey_host", rc);
    for (size_t i = 0; i < n; i++) ok[i] = v[i] == 1;
    free(buf);
}

void check_tx_sigs_bip143_batch(const void *sv_tx_array, const u8 *scripts, size_t scripts_len,
                                const struct pubkey *key, const struct bitcoin_signature *sigs, size_t n, bool *ok) {
    if (n == 0) return;
    sv_tx *txs = (sv_tx *)malloc(n * sizeof(sv_tx));
    u8 *buf = (u8 *)malloc(n * (64 + 64 + 1));
    if (!txs || !buf) die("malloc", -3);
    memcpy(txs, sv_tx_array, n * sizeof(sv_tx));
    u8 *xy = buf, *sig = buf + 64 * n, *v = sig + 64 * n;
    for (size_t i = 0; i < n; i++) {
        txs[i].sighash_type = (uint32_t)sigs[i].sighash_type; /* the type committed to is the signature's */
        pubkey_to_xy(xy + 64 * i, &key->pubkey);
        sig_to_wire(sig + 64 * i, &sigs[i].s);
    }
    int rc = sv_verify_tx_host(ctx(), SV_KIND_ECDSA_XY, txs, scripts, scripts_len, xy, sig, n, v, NULL);
    if (rc != SV_OK) die("sv_verify_tx_host", rc);
    for (size_t i = 0; i < n; i++) {
        /* check_tx_sig's gate (signature.c:206-211); a witness script is always present on this path */
        bool type_ok = sigs[i].sighash_type == SIGHASH_ALL ||
                       (int)sigs[i].sighash_type == (SIGHASH_SINGLE | SIGHASH_ANYONECANPAY);
        ok[i] = type_ok && v[i] == 1;
    }
    free(txs);
    free(buf);
}

/* ---- gossip: the raw wire messages go to the device as one blob; the DEVICE slices them the way
 * gossipd/sigcheck.c does (k_gossip_slice), hashes the signed regions and verifies (sv_verify_gossip_host) ---- */
static void gossip_batch(const u8 *const *msgs, const size_t *lens, size_t n, const struct node_id *signers,
                         uint16_t want_type, int *status) {
    if (n == 0) return;
    size_t total = 0;
    for (size_t i = 0; i < n; i++) total += lens[i];
    u8 *blob = (u8 *)malloc(total ? total : 1);
    uint64_t *off = (uint64_t *)malloc(n * sizeof(uint64_t));
    uint32_t *len = (uint32_t *)malloc(n * sizeof(uint32_t));
    if (!blob || !off || !len) die("malloc", -3);
    size_t t = 0;
    for (size_t i = 0; i < n; i++) {
        off[i] = t;
        len[i] = (uint32_t)lens[i];
        memcpy(blob + t, msgs[i], lens[i]);
        t += lens[i];
    }
    int rc = sv_verify_gossip_host(ctx(), blob, total, off, len, n, signers ? signers[0].k : NULL, status);
    if (rc != SV_OK) die("sv_verify_gossip_host", rc);
    for (size_t i = 0; i < n; i++) /* this entry point is typed: a message of another kind is malformed here */
        if (lens[i] < 2 || (uint16_t)((msgs[i][0] << 8) | msgs[i][1]) != want_type) status[i] = -1;
    free(blob); free(off); free(len);
}

void sigcheck_channel_announcement_batch(const u8 *const *msgs, const size_t *lens, size_t n, int *status) {
    gossip_batch(msgs, lens, n, NULL, 256, status);
}
void sigcheck_node_announcement_batch(const u8 *const *msgs, const size_t *lens, size_t n, int *status) {
    gossip_batch(msgs, lens, n, NULL, 257, status);
}
void sigcheck_channel_update_batch(const u8 *const *msgs, const size_t *lens, const struct node_id *signers,
                                   size_t n, int *status) {
    gossip_batch(msgs, lens, n, signers, 258, status); /* struct node_id is exactly 33 bytes: signers[] is the packed array */
}
