// verify.cuh — one signature verification, split the way the engine's kernels run it:
//
//   scalar side  (K_prep) : parse/range-check (r,s), s^-1 (amortised over a batch of 32 with
//                           Montgomery's trick), u1 = m/s, u2 = r/s, GLV split of u2, window
//                           recoding  ->  128-byte sv_work record
//   curve side   (K_main) : key decode (33-byte compressed / 64-byte x|y / 32-byte x-only),
//                           per-key odd-multiples table, fixed-window ladder for u2*Q, fixed-base
//                           comb for u1*G, final x (and y-parity) comparison  ->  verdict
//
// Accept/reject rules are those of the reference, bit for bit (SURVEY.md Appendix A):
//   ECDSA  : secp256k1_ecdsa_signature_parse_compact (secp256k1.c:377-396) + secp256k1_ecdsa_verify
//            (secp256k1.c:442-456) + secp256k1_ecdsa_sig_verify (ecdsa_impl.h:195-264)
//            + secp256k1_eckey_pubkey_parse (eckey_impl.h:17-35)
//   Schnorr: secp256k1_xonly_pubkey_parse (modules/extrakeys/main_impl.h:23-43)
//            + secp256k1_schnorrsig_verify (modules/schnorrsig/main_impl.h:219-265)
// The double-scalar multiplication is NOT the reference's Strauss-wNAF (ecmult_impl.h:234-341):
// wNAF digit positions are data dependent, which would make the 32 lanes of a warp add at
// different ladder steps.  Here every lane executes the same schedule:
//   u2*Q : GLV split (same endomorphism as scalar_impl.h:138-176), both halves forced odd, regular
//          signed-odd-digit recoding with 4-bit windows -> 33 windows, 128 doublings, 65 mixed adds
//          against an 8-entry odd-multiples table kept effective-affine by the isomorphism trick of
//          ecmult_impl.h:73-115;
//   u1*G : signed 16-bit comb over a precomputed affine table of d*2^(16 i)*G (gtable.cuh): 16 mixed
//          adds, no doublings.  (Reference: 2 x 8192-entry wNAF tables, precomputed_ecmult.c.)
#pragma once
#include "ge.cuh"
#include "sc.cuh"
#include "sha256.cuh"

#define SV_KIND_ECDSA33 0   // msg32 | pub33 (02/03 || x) | sig64 (r||s)
#define SV_KIND_ECDSA_XY 1  // msg32 | pubxy64 (x || y)   | sig64 (r||s)      (pre-decompressed key)
#define SV_KIND_SCHNORR 2   // msg32 | xonly32            | sig64 (R.x||s)    BIP-340
#define SV_KIND_ECDSA33_NS 3  // internal: kind 0 through the flow that never takes the square root (see below)
#define SV_KIND_SCHNORR_NS 4  // internal: kind 2 likewise
#define SV_KIND_RECOVER 5     // internal: msg32 | recid (1 byte in the key slot) | sig64 (r||s) -> public key (see "recovery")

// G comb table geometry: rows 0..14 hold d*B_i for d = 1..32768, row 15 holds d = 1..65536
#define SV_GT_ROW 32768
#define SV_GT_ENTRIES (15 * SV_GT_ROW + 65536)

struct alignas(16) ge_mem {  // affine point as stored in HBM: 64 bytes, 4 x LDG.128
    u32 x[8], y[8];
};
struct alignas(16) qtab_entry {  // per-verification odd-multiples scratch entry (96 bytes)
    u32 x[8], y[8], h[8];
};

SV_HD void ge_from_mem(ge& r, const ge_mem* p) {
#if SV_DEVICE_CODE
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = q[0], b = q[1], c = q[2], d = q[3];
    r.x.v[0] = a.x; r.x.v[1] = a.y; r.x.v[2] = a.z; r.x.v[3] = a.w;
    r.x.v[4] = b.x; r.x.v[5] = b.y; r.x.v[6] = b.z; r.x.v[7] = b.w;
    r.y.v[0] = c.x; r.y.v[1] = c.y; r.y.v[2] = c.z; r.y.v[3] = c.w;
    r.y.v[4] = d.x; r.y.v[5] = d.y; r.y.v[6] = d.z; r.y.v[7] = d.w;
#else
    for (int i = 0; i < 8; i++) { r.x.v[i] = p->x[i]; r.y.v[i] = p->y[i]; }
#endif
}
SV_HD void ge_to_mem(ge_mem* p, const ge& a) {
#if SV_DEVICE_CODE
    uint4* q = reinterpret_cast<uint4*>(p);
    q[0] = make_uint4(a.x.v[0], a.x.v[1], a.x.v[2], a.x.v[3]);
    q[1] = make_uint4(a.x.v[4], a.x.v[5], a.x.v[6], a.x.v[7]);
    q[2] = make_uint4(a.y.v[0], a.y.v[1], a.y.v[2], a.y.v[3]);
    q[3] = make_uint4(a.y.v[4], a.y.v[5], a.y.v[6], a.y.v[7]);
#else
    for (int i = 0; i < 8; i++) { p->x[i] = a.x.v[i]; p->y[i] = a.y.v[i]; }
#endif
}
SV_HD void fe_from_words(fe& r, const u32* p) {
#if SV_DEVICE_CODE
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = q[0], b = q[1];
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
    r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
#else
    for (int i = 0; i < 8; i++) r.v[i] = p[i];
#endif
}
SV_HD void fe_to_words(u32* p, const fe& a) {
#if SV_DEVICE_CODE
    uint4* q = reinterpret_cast<uint4*>(p);
    q[0] = make_uint4(a.v[0], a.v[1], a.v[2], a.v[3]);
    q[1] = make_uint4(a.v[4], a.v[5], a.v[6], a.v[7]);
#else
    for (int i = 0; i < 8; i++) p[i] = a.v[i];
#endif
}

// =================================================================================================
// scalar side
// =================================================================================================

// ECDSA: parse (r,s) and the message hash.  Returns false (verdict 0) for r >= n, s >= n
// (parse_compact, secp256k1.c:388-392), r == 0, s == 0 (ecdsa_impl.h:204), s > n/2
// (secp256k1.c:451).  The message is reduced mod n and never rejected (secp256k1.c:449).
SV_HD bool ecdsa_parse(sc& r, sc& s, sc& m, const u8* sig64, const u8* msg32, bool* parsed = nullptr) {
    bool ovr, ovs;
    sc_set_b32(r, sig64, &ovr);
    sc_set_b32(s, sig64 + 32, &ovs);
    sc_set_b32(m, msg32, nullptr);
    if (parsed) *parsed = !ovr && !ovs;  // what CLN's wire layer checks (wire/fromwire.c:188-199)
    bool ok = !ovr && !ovs && !sc_is_zero(r) && !sc_is_zero(s) && !sc_is_high(s);
    return ok;
}

SV_HD void work_set_invalid(sv_work& w) {
    SV_UNROLL
    for (int i = 0; i < 5; i++) { w.k1[i] = 0; w.k2[i] = 0; w.pad[i] = 0; }
    w.k1[0] = 1;
    w.k2[0] = 1;
    SV_UNROLL
    for (int i = 0; i < 16; i++) w.gd[i] = 0;
    w.flags = 0;
}

// ECDSA: given s^-1, finish the record: u1 = m/s, u2 = r/s (ecdsa_impl.h:209-211)
SV_HD void ecdsa_finish_prep(sv_work& w, bool ok, const sc& r, const sc& m, const sc& sinv, bool parsed = true) {
    if (!ok) {
        work_set_invalid(w);
        w.flags = parsed ? SV_WF_PARSED : 0u;
        return;
    }
    sc u1, u2;
    sc_mul(u1, sinv, m);
    sc_mul(u2, sinv, r);
    SV_UNROLL
    for (int i = 0; i < 5; i++) w.pad[i] = 0;
    sc_prepare_u2(w, u2);
#ifdef SV_COMB_SMEM
    sc_prepare_u1_smem(w, u1);
#else
    sc_prepare_u1(w, u1);
#endif
    // second x candidate r + n exists iff r < p - n (ecdsa_impl.h:253-259; constant :32-34)
    const u32 pmn[8] = {0x2FC9BAEEu, 0x402DA172u, 0x50B75FC4u, 0x45512319u, 0x00000001u, 0, 0, 0};
    u32 t[8];
    u32 bw = u256_sub(t, r.v, pmn);
    w.flags = SV_WF_VALID | SV_WF_PARSED | (bw ? SV_WF_R_PLUS_N : 0u);
}

// BIP-340: R = s*G + (-e)*P with e = H_tag(r || P.x || m) mod n.   Rejects r >= p
// (main_impl.h:235) and s >= n (:239-242).
SV_HD void schnorr_prep(sv_work& w, const u8* sig64, const u8* xonly32, const u8* msg32) {
    fe rx;
    bool ovs;
    sc s, e, ne;
    bool ok = fe_set_b32(rx, sig64);
    sc_set_b32(s, sig64 + 32, &ovs);
    ok = ok && !ovs;
    if (!ok) {
        work_set_invalid(w);
        return;
    }
    u8 h[32];
    sha256_bip340_challenge(h, sig64, xonly32, msg32);
    sc_set_b32(e, h, nullptr);
    sc_negate(ne, e);
    SV_UNROLL
    for (int i = 0; i < 5; i++) w.pad[i] = 0;
    sc_prepare_u2(w, ne);
#ifdef SV_COMB_SMEM
    sc_prepare_u1_smem(w, s);
#else
    sc_prepare_u1(w, s);
#endif
    w.flags = SV_WF_VALID;
}

// Montgomery's trick: invert n (<= SV_PREP_BATCH) non-zero scalars with ONE exponentiation.
#define SV_PREP_BATCH 32
SV_HD void sc_batch_inverse(sc* v, int n) {
    sc pre[SV_PREP_BATCH];
    sc acc;
    pre[0] = v[0];
    for (int i = 1; i < n; i++) sc_mul(pre[i], pre[i - 1], v[i]);
    sc_inverse(acc, pre[n - 1]);
    for (int i = n - 1; i > 0; i--) {
        sc t;
        sc_mul(t, acc, pre[i - 1]);  // = 1 / v[i]
        sc_mul(acc, acc, v[i]);
        v[i] = t;
    }
    v[0] = acc;
}

// =================================================================================================
// curve side
// =================================================================================================

// decode the public key of item `kind`; false -> verdict 0
SV_HD bool key_decode(ge& Q, int kind, const u8* key) {
    // No early exits: every lane runs the same instruction stream (an invalid key just carries a false
    // flag and garbage coordinates through the ladder), so CTA-wide barriers stay legal and nothing is
    // lost — in SIMT a lane that leaves early saves no time while its warp keeps going.
    if (kind == SV_KIND_ECDSA33) {
        // eckey_impl.h:17-20: prefix must be 02/03, x < p, x^3+7 a residue
        u8 pfx = key[0];
        fe x;
        bool ok = (pfx == 2 || pfx == 3);
        ok = fe_set_b32(x, key + 1) && ok;
        return ge_set_xo(Q, x, pfx == 3) && ok;
    } else if (kind == SV_KIND_ECDSA_XY) {
        // eckey_impl.h:21-33 (65-byte form without the 04 prefix): x,y < p and on the curve
        bool ok = fe_set_b32(Q.x, key);
        ok = fe_set_b32(Q.y, key + 32) && ok;
        return ge_is_on_curve(Q) && ok;
    } else {
        // extrakeys/main_impl.h:32-38: x < p, lift to the even-y point
        fe x;
        bool ok = fe_set_b32(x, key);
        return ge_set_xo(Q, x, false) && ok;
    }
}

// bits [4i+1, 4i+5) of a 160-bit magnitude, i <= 31 (highest bit touched is 128, so the sign bit
// kept in bit 159 never enters a window); read straight from the work record
SV_HD u32 window4(const u32* mag, int i) {
    int off = 4 * i + 1;
    int l = off >> 5, sh = off & 31;
    u64 two = ((u64)mag[l + 1] << 32) | mag[l];  // l <= 3
    return (u32)(two >> sh) & 15u;
}

// Build the effective-affine table of {1,3,...,15}*Q in `tab` (x,y valid on return) and return
// the common Z of the table in true curve coordinates (zc).  124 field mul/sqr.
SV_HD void qtable_build(qtab_entry* tab, fe& zc, const ge& Q, unsigned sync_threads = 0) {
    gej D, acc;
    gej_set_ge(D, Q);
    gej_double(D, D);  // 2Q = (Xd, Yd, Zd);  on the curve scaled by c = Zd it is the affine point (Xd, Yd)
    fe c2, c3;
    fe_sqr(c2, D.z);
    fe_mul(c3, c2, D.z);
    ge d_aff, q1;
    d_aff.x = D.x;
    d_aff.y = D.y;
    fe_mul(q1.x, Q.x, c2);  // Q on the scaled curve
    fe_mul(q1.y, Q.y, c3);
    gej_set_ge(acc, q1);
    fe_to_words(tab[0].x, q1.x);
    fe_to_words(tab[0].y, q1.y);
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
    for (int k = 1; k < 8; k++) {
        fe h;
        SV_SYNC(sync_threads);
        gej_add_ge(acc, acc, d_aff, &h);  // (2k+1)Q ; never exceptional for a point of prime order > 15
        fe_to_words(tab[k].x, acc.x);
        fe_to_words(tab[k].y, acc.y);
        fe_to_words(tab[k].h, h);
    }
    fe_mul(zc, acc.z, D.z);
    // bring entries 6..0 to the Z of entry 7:  ratio_k = prod_{j=k+1..7} h_j
    fe zr;
    fe_from_words(zr, tab[7].h);
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
    for (int k = 6; k >= 0; k--) {
        fe zr2, zr3, t;
        fe_sqr(zr2, zr);
        fe_mul(zr3, zr2, zr);
        fe_from_words(t, tab[k].x);
        fe_mul(t, t, zr2);
        fe_to_words(tab[k].x, t);
        fe_from_words(t, tab[k].y);
        fe_mul(t, t, zr3);
        fe_to_words(tab[k].y, t);
        if (k > 0) {
            fe_from_words(t, tab[k].h);
            fe_mul(zr, zr, t);
        }
    }
    // the ratio slots are free now: store beta*x there, the x coordinate of lambda*P (endomorphism half)
    fe beta;
    SV_UNROLL
    for (int i = 0; i < 8; i++) beta.v[i] = GE_BETA[i];
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
    for (int k = 0; k < 8; k++) {
        fe t;
        fe_from_words(t, tab[k].x);
        fe_mul(t, t, beta);
        fe_to_words(tab[k].h, t);
    }
}

// fetch table entry for window value v (0..15) of a scalar with sign `sneg`; lam -> apply beta
SV_HD void qtable_fetch(ge& p, const qtab_entry* tab, u32 v, u32 sneg, bool lam) {
    u32 dneg = (v < 8) ? 1u : 0u;
    u32 idx = dneg ? (7u - v) : (v - 8u);
    fe_from_words(p.x, lam ? tab[idx].h : tab[idx].x);  // h slot holds beta*x
    fe_from_words(p.y, tab[idx].y);
    if (dneg ^ sneg) fe_neg(p.y, p.y);
}

// R = u2*Q in true Jacobian coordinates, given a ready odd-multiples table of Q (common Z = zc): the joint ladder over
// both GLV halves (128 doublings, 2 x 33 mixed additions)
SV_HD void ecmult_ladder_q(gej& R, const sv_work* w, const qtab_entry* tab, const fe& zc, unsigned sync_threads = 0) {
    const u32* m1 = w->k1;
    const u32* m2 = w->k2;
    u32 t1 = m1[4], t2 = m2[4];
    u32 s1 = t1 >> 31, s2 = t2 >> 31;
    ge p;
    // top window (i = 32): digit = 2*(mag >> 129) + 1, always positive
    {
        u32 v1 = (t1 >> 1) & 7u, v2 = (t2 >> 1) & 7u;
        qtable_fetch(p, tab, v1 + 8u, s1, false);
        gej_set_ge(R, p);
        qtable_fetch(p, tab, v2 + 8u, s2, true);
        gej_add_ge(R, R, p);
    }
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
    for (int i = 31; i >= 0; i--) {
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
#if defined(SV_SYNC_LEVEL) && SV_SYNC_LEVEL < 2
#ifndef SV_SYNC_WINDOWS
#define SV_SYNC_WINDOWS 1
#endif
        if (i % SV_SYNC_WINDOWS == 0) SV_SYNC(sync_threads);  // one re-convergence point per SV_SYNC_WINDOWS windows
#endif
        for (int j = 0; j < 4; j++) {
#if !defined(SV_SYNC_LEVEL) || SV_SYNC_LEVEL >= 2
            SV_SYNC(sync_threads);
#endif
            gej_double(R, R);
        }
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
        for (int half = 0; half < 2; half++) {
            u32 v = half ? window4(m2, i) : window4(m1, i);
#if !defined(SV_SYNC_LEVEL) || SV_SYNC_LEVEL >= 2
            SV_SYNC(sync_threads);
#endif
            qtable_fetch(p, tab, v, half ? s2 : s1, half != 0);
            gej_add_ge(R, R, p);
        }
    }
    // leave the scaled curve: true Z = Z * zc
    fe_mul(R.z, R.z, zc);
}

// R += u1*G through the fixed-base comb (16 mixed additions against the 34 MiB table)
SV_HD void ecmult_comb_add(gej& R, const sv_work* w, const ge_mem* gtab, unsigned sync_threads = 0) {
    ge p;
#if defined(SV_COMB_SMEM) && SV_DEVICE_CODE
    // VARIANT: 8-bit GLV comb against the 131 KB table staged in shared memory (k_main copies it in with one bulk copy):
    // 2 x 17 windows -> up to 34 mixed additions and a beta multiplication for each lambda-half point
    {
        extern __shared__ __align__(16) unsigned char sv_smem_raw[];
        const ge_mem* t8 = reinterpret_cast<const ge_mem*>(sv_smem_raw);
        fe beta;
        SV_UNROLL
        for (int i = 0; i < 8; i++) beta.v[i] = GE_BETA[i];
        const u32 top = w->pad[0];
#pragma unroll 1
        for (int row = 0; row < 17; row++) {
            SV_SYNC(sync_threads);
#pragma unroll 1
            for (int half = 0; half < 2; half++) {
                int d;
                if (row < 16) d = half ? (int)(short)((u32)w->gd[row] >> 16) : (int)(short)((u32)w->gd[row] & 0xFFFFu);
                else d = (int)(signed char)((top >> (8 * half)) & 0xFFu);
                u32 sneg = (top >> (16 + half)) & 1u;
                if (d != 0) {
                    u32 a = (u32)(d < 0 ? -d : d);
                    ge_from_mem(p, t8 + (size_t)row * 128 + (a - 1));
                    if (half) fe_mul(p.x, p.x, beta);
                    if ((d < 0) != (sneg != 0)) fe_neg(p.y, p.y);
                    gej_add_ge(R, R, p);
                }
            }
        }
    }
#else
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
    for (int row = 0; row < 16; row++) {
        int d = w->gd[row];
        SV_SYNC(sync_threads);
        if (d != 0) {
            u32 a = (u32)(d < 0 ? -d : d);
            ge_from_mem(p, gtab + (size_t)row * SV_GT_ROW + (a - 1));
            if (d < 0) fe_neg(p.y, p.y);
            gej_add_ge(R, R, p);
        }
    }
#endif
}

// R = u1*G + u2*Q in true Jacobian coordinates
SV_HD void ecmult_ladder(gej& R, const sv_work* w, const ge_mem* gtab, const qtab_entry* tab, const fe& zc,
                         unsigned sync_threads = 0) {
    ecmult_ladder_q(R, w, tab, zc, sync_threads);
    ecmult_comb_add(R, w, gtab, sync_threads);
}

SV_HD void ecmult_uniform(gej& R, const sv_work* w, const ge& Q, const ge_mem* gtab, qtab_entry* tab,
                          unsigned sync_threads = 0) {
    fe zc;
    qtable_build(tab, zc, Q, sync_threads);
    ecmult_ladder(R, w, gtab, tab, zc, sync_threads);
}

SV_HD u32 ecdsa_final(const gej& R, const u8* sig64, u32 flags);

// ---- one key, many signatures (channeld's HTLC loop, SURVEY.md §8a a16 / §8f N3): the key is decoded and its
// odd-multiples table built ONCE (k_sharedkey_build); every verification then skips the square root (267 field mults)
// and the table build (132): ~18 % less work per signature.
struct alignas(16) sv_shared_key {
    qtab_entry tab[8];
    u32 zc[8];
    u32 ok, pad[3];
};
SV_HD void sharedkey_build(sv_shared_key* out, int kind, const u8* key, unsigned sync_threads = 0) {
    ge Q;
    bool ok = key_decode(Q, kind, key);
    fe zc;
    qtable_build(out->tab, zc, Q, sync_threads);
    fe_to_words(out->zc, zc);
    out->ok = ok ? 1u : 0u;
}
SV_HD u32 verify_curve_side_shared(const sv_work* w, const u8* sig64, const ge_mem* gtab, const sv_shared_key* sk,
                                   unsigned sync_threads = 0) {
    u32 flags = w->flags;
    bool ok = (flags & SV_WF_VALID) != 0 && sk->ok != 0;
    fe zc;
    fe_from_words(zc, sk->zc);
    gej R;
    ecmult_ladder(R, w, gtab, sk->tab, zc, sync_threads);
    u32 v = ecdsa_final(R, sig64, flags);
    return ok ? v : 0u;
}

// final comparison, ECDSA: x(R) mod n == r without leaving Jacobian coordinates
// (ecdsa_impl.h:229-264; secp256k1_gej_eq_x_var group_impl.h:396-404)
SV_HD u32 ecdsa_final(const gej& R, const u8* sig64, u32 flags) {
    if (R.inf) return 0;
    fe xr, zz, t;
    fe_set_b32(xr, sig64);  // r < n < p
    fe_sqr(zz, R.z);
    fe_mul(t, xr, zz);
    if (fe_equal(t, R.x)) return 1;
    if (flags & SV_WF_R_PLUS_N) {
        fe nn;
        SV_UNROLL
        for (int i = 0; i < 8; i++) nn.v[i] = SC_N[i];
        u256_add(xr.v, xr.v, nn.v);  // r + n < p: no wrap
        fe_mul(t, xr, zz);
        if (fe_equal(t, R.x)) return 1;
    }
    return 0;
}

// final comparison, BIP-340: R finite, y(R) even, x(R) == r  (main_impl.h:255-264)
SV_HD u32 schnorr_final(const gej& R, const u8* sig64, bool var_time_inverse = false) {
    if (R.inf) return 0;
    fe zi, rx;
    ge a;
    if (var_time_inverse) fe_inv_var(zi, R.z); else fe_inv(zi, R.z);
    ge_set_gej_zinv(a, R, zi);
    fe_normalize(a.y);
    if (fe_is_odd(a.y)) return 0;
    fe_set_b32(rx, sig64);
    return fe_equal(rx, a.x) ? 1u : 0u;
}

// BIP-340 needs the affine R (y parity): one field inversion per signature.  Instead of inverting inside the
// ladder kernel, it parks R = (X,Y,Z) in the (now dead) 128-byte work record and a small second kernel inverts
// 16 Z's at a time with Montgomery's trick (3 mults per signature + 1/16 of a Fermat exponentiation).
struct alignas(16) sv_jac {
    u32 x[8], y[8], z[8];
    u32 inf, ok, pad[6];
};
#define SV_FINAL_BATCH 16

SV_HD void schnorr_park(sv_jac* out, const gej& R, bool ok) {
    fe_to_words(out->x, R.x);
    fe_to_words(out->y, R.y);
    fe_to_words(out->z, R.z);
    out->inf = R.inf;
    out->ok = ok ? 1u : 0u;
}

// verdicts for cnt (<= SV_FINAL_BATCH) consecutive parked results
SV_HD void schnorr_final_batch(u8* verdict, const sv_jac* jac, const u8* sig64, int cnt) {
    fe pre[SV_FINAL_BATCH];
    fe acc, one;
    fe_set_u32(one, 1);
    for (int i = 0; i < cnt; i++) {
        fe z;
        fe_from_words(z, jac[i].z);
        bool usable = jac[i].ok && !jac[i].inf && !fe_is_zero(z);
        if (!usable) z = one;
        if (i == 0) pre[0] = z; else fe_mul(pre[i], pre[i - 1], z);
    }
    fe_inv(acc, pre[cnt - 1]);
    for (int i = cnt - 1; i >= 0; i--) {
        fe z, zi;
        fe_from_words(z, jac[i].z);
        bool usable = jac[i].ok && !jac[i].inf && !fe_is_zero(z);
        if (!usable) z = one;
        if (i > 0) {
            fe_mul(zi, acc, pre[i - 1]);
            fe_mul(acc, acc, z);
        } else {
            zi = acc;
        }
        gej R;
        fe_from_words(R.x, jac[i].x);
        fe_from_words(R.y, jac[i].y);
        ge a;
        ge_set_gej_zinv(a, R, zi);
        fe_normalize(a.y);
        fe rx;
        fe_set_b32(rx, sig64 + 64 * i);
        bool good = usable && !fe_is_odd(a.y) && fe_equal(rx, a.x);  // main_impl.h:255-264
        verdict[i] = good ? 1 : 0;
    }
}

// ---- public-key recovery (secp256k1_ecdsa_recover, modules/recovery/main_impl.h:87-156) --------------------------------
// Q = (-m/r)*G + (s/r)*R with R = lift(r (+ n if recid & 2)), y(R) odd iff recid & 1.  The same split as a verification:
// the scalar side writes u1 = -m/r into the comb digits and u2 = s/r into the GLV halves, the curve side lifts R (one
// square root), runs the same double-scalar multiplication and parks Q; the affine key needs one field inversion, batched
// 16 at a time like the BIP-340 final step.  Outcomes per item:
//   -1  encoding refused: r >= n, s >= n (recoverable_signature_parse_compact, main_impl.h:38-57) or recid > 3
//    0  recovery failed, key all zero: r == 0, s == 0, recid & 2 with r >= p - n, no curve point with x = r (+ n), Q = inf
//    1  key = affine x || y of Q, big-endian.  No low-S rule: a high s recovers.
#define SV_RECOVER_REFUSED 0xFFu  // the status byte of outcome -1 (int8_t -1)

// scalar side of one item, given 1/r (r != 0) or anything (invalid item).  ok: r, s in range and non-zero, recid <= 3.
SV_HD void recover_parse(sc& r, sc& s, sc& m, bool& ok, bool& parsed, const u8* sig64, const u8* msg32, u32 recid) {
    bool ovr, ovs;
    sc_set_b32(r, sig64, &ovr);
    sc_set_b32(s, sig64 + 32, &ovs);
    sc_set_b32(m, msg32, nullptr);  // m mod n, never rejected (main_impl.h:138)
    parsed = !ovr && !ovs && recid <= 3u;
    ok = parsed && !sc_is_zero(r) && !sc_is_zero(s);  // ecdsa_sig_recover, main_impl.h:93-95
}
SV_HD void recover_finish_prep(sv_work& w, bool ok, bool parsed, const sc& r, const sc& s, const sc& m, const sc& rinv) {
    if (!ok) {
        work_set_invalid(w);
        w.flags = parsed ? SV_WF_PARSED : 0u;
        return;
    }
    sc u1, u2;
    sc_mul(u1, rinv, m);
    sc_negate(u1, u1);  // -m/r  (main_impl.h:113-114)
    sc_mul(u2, rinv, s);  // s/r (:115)
    SV_UNROLL
    for (int i = 0; i < 5; i++) w.pad[i] = 0;
    sc_prepare_u2(w, u2);
#ifdef SV_COMB_SMEM
    sc_prepare_u1_smem(w, u1);
#else
    sc_prepare_u1(w, u1);
#endif
    const u32 pmn[8] = {0x2FC9BAEEu, 0x402DA172u, 0x50B75FC4u, 0x45512319u, 0x00000001u, 0, 0, 0};  // p - n
    u32 t[8];
    u32 bw = u256_sub(t, r.v, pmn);
    w.flags = SV_WF_VALID | SV_WF_PARSED | (bw ? SV_WF_R_PLUS_N : 0u);
}

// R from r and the recovery id, without the range check of r + n (the scalar side's SV_WF_R_PLUS_N, which the caller
// ANDs in): false if x^3 + 7 is not a square (main_impl.h:97-107).  No early exit: see key_decode.
SV_HD bool recover_lift(ge& R, const u8* sig64, u32 recid) {
    fe x;
    fe_set_b32(x, sig64);  // r < n < p for every item that can succeed
    if (recid & 2u) {
        fe nn;
        SV_UNROLL
        for (int i = 0; i < 8; i++) nn.v[i] = SC_N[i];
        u256_add(x.v, x.v, nn.v);  // r + n < p when it counts
    }
    return ge_set_xo(R, x, (recid & 1u) != 0);
}
SV_HD bool recover_lift_allowed(u32 flags, u32 recid) {
    return (flags & SV_WF_VALID) != 0 && (!(recid & 2u) || (flags & SV_WF_R_PLUS_N) != 0);
}

// Q parked in place of the work record: ok = a point may come out, pad[0] = the encoding parsed (status 0 rather than -1)
SV_HD void recover_park(sv_jac* out, const gej& Q, bool ok, bool parsed) {
    schnorr_park(out, Q, ok);
    out->pad[0] = parsed ? 1u : 0u;
}

SV_HD void recover_emit(u8* xy64, u8* status, const ge* a, bool parsed) {
    if (a) {
        fe_get_b32(xy64, a->x);
        fe_get_b32(xy64 + 32, a->y);
        *status = 1;
    } else {
        for (int k = 0; k < 64; k++) xy64[k] = 0;  // main_impl.h:150-156
        *status = parsed ? 0u : SV_RECOVER_REFUSED;
    }
}

// keys and statuses for cnt (<= SV_FINAL_BATCH) consecutive parked results: one Fermat inversion for all their Z's
SV_HD void recover_final_batch(u8* xy64, u8* status, const sv_jac* jac, int cnt) {
    fe pre[SV_FINAL_BATCH];
    fe acc, one;
    fe_set_u32(one, 1);
    for (int i = 0; i < cnt; i++) {
        fe z;
        fe_from_words(z, jac[i].z);
        bool usable = jac[i].ok && !jac[i].inf && !fe_is_zero(z);
        if (!usable) z = one;
        if (i == 0) pre[0] = z; else fe_mul(pre[i], pre[i - 1], z);
    }
    fe_inv(acc, pre[cnt - 1]);
    for (int i = cnt - 1; i >= 0; i--) {
        fe z, zi;
        fe_from_words(z, jac[i].z);
        bool usable = jac[i].ok && !jac[i].inf && !fe_is_zero(z);
        if (!usable) z = one;
        if (i > 0) {
            fe_mul(zi, acc, pre[i - 1]);
            fe_mul(acc, acc, z);
        } else {
            zi = acc;
        }
        gej Q;
        fe_from_words(Q.x, jac[i].x);
        fe_from_words(Q.y, jac[i].y);
        ge a;
        ge_set_gej_zinv(a, Q, zi);
        recover_emit(xy64 + 64 * i, status + i, usable ? &a : nullptr, jac[i].pad[0] != 0);
    }
}

// whole curve side for one item
SV_HD u32 verify_curve_side(int kind, const sv_work* w, const u8* key, const u8* sig64, const ge_mem* gtab,
                            qtab_entry* tab, bool* key_ok = nullptr, unsigned sync_threads = 0) {
    u32 flags = w->flags;
    bool ok = (flags & SV_WF_VALID) != 0;  // an invalid record carries harmless dummy scalars (k1 = k2 = 1, u1 = 0)
    ge Q;
    bool kd = key_decode(Q, kind, key);
    if (key_ok) *key_ok = kd;
    ok = kd && ok;
    gej R;
    ecmult_uniform(R, w, Q, gtab, tab, sync_threads);
    u32 v = (kind == SV_KIND_SCHNORR) ? schnorr_final(R, sig64) : ecdsa_final(R, sig64, flags);
    return ok ? v : 0u;
}

// ---- compressed-key ECDSA without the square root -------------------------------------------------------------------
// Decompressing a 33-byte key costs a square root (254 squarings + 13 multiplications, 10 % of a verification).  It can be
// traded for ~50 multiplications by never materialising y:  with c = x^3 + 7 and y the (unknown) root of c,
//   * phi: (X, Y) -> (y^2 X, y^3 Y) maps the curve onto  E': Y^2 = X^3 + 7 c^3  and sends Q = (x, y) to Q' = (c x, c^2),
//     which needs no y.  The doubling / addition formulas never use the curve constant, so table build and GLV ladder run
//     on E' unchanged (the endomorphism is still X -> beta X) and give S' = u2*Q' = (X1, Y1, Zs);
//   * pulled back, u2*Q = (X1, Y1, y*Zs) on the real curve: y only scales Z.  Adding T = u1*G = (X2, Y2, Z2) with the
//     Jacobian addition formulas and collecting powers of y (y^2 = c) gives  X3 = A - y*B  and  Z3^2 = c*z3^2  with A, B,
//     z3 free of y, so the ECDSA test  X3 == r * Z3^2  reads   y * B == A - r*c*z3^2 =: D ;
//   * it is linear in y: the signature is valid iff  y = D/B  is THE root the key names, i.e. (D/B)^2 == c and the parity
//     of D/B equals the prefix bit.  For an invalid key (c a non-residue) no value squares to c: verdict 0, as
//     secp256k1_eckey_pubkey_parse refusing the key (eckey_impl.h:17-20, group_impl.h:334-346).
// The division is batched in k_final_ecdsa33 (Montgomery's trick over 16 signatures).  Rare configurations the linear form
// does not cover (u1*G or u2*Q at infinity, equal x coordinates, B == 0, the r + n candidate of ecdsa_impl.h:250-262) are
// re-verified there by the plain path with the real square root, so verdicts stay bit-exact.
#define SV_NS_PENDING 2u  // D, B, c parked: k_final_ecdsa33 decides
#define SV_NS_EXACT 4u    // work record left intact: k_final_ecdsa33 runs the plain path
struct alignas(16) sv_ns_park {
    u32 d[8], b[8], c[8], pad[8];
};

// The linear form itself.  S = (X1, Y1, y*Zs) with y^2 = c, T = (X2, Y2, Z2), both finite.  Jacobian addition S + T with the
// powers of y collected:  X3 = A - y*B,  Z3 = y*z3,  so  x(S + T) == r  <=>  y*B == D := A - r*c*z3^2.
// Returns true when the form does not apply (equal x coordinates, or B == 0): the caller falls back to the plain path.
// With ext != nullptr also  Y3 = E + y*F  is worked out and  ext[0] = N = E*B + F*D,  ext[1] = CG = c*z3^3  (BIP-340:
// y(S + T) = N / (D*CG) once y = D/B).
SV_HD bool ns_linear_form(fe& D, fe& B, const fe& X1, const fe& Y1, const fe& Zs, const gej& T, const fe& c, const fe& rfe,
                          fe* ext = nullptr) {
    fe z2z2, t, U1, S1, czs2, s2p, H, z3, A, HH, V, K, W0;
    fe_sqr(z2z2, T.z);
    fe_mul(U1, X1, z2z2);            // U1 = X1 Z2^2
    fe_mul(t, T.z, z2z2);
    fe_mul(S1, Y1, t);               // S1 = Y1 Z2^3
    fe_sqr(t, Zs);
    fe_mul(czs2, c, t);              // (y Zs)^2
    fe_mul(H, T.x, czs2);            // U2 = X2 (y Zs)^2
    fe_sub(H, H, U1);                // H = U2 - U1
    fe_mul(t, Zs, czs2);
    fe_mul(s2p, T.y, t);             // S2 = y * s2p,  s2p = Y2 c Zs^3
    bool exact = fe_is_zero(H);      // equal x coordinates: doubling or infinity, depending on the sign of y
    fe_mul(z3, H, Zs);
    fe_mul(z3, z3, T.z);             // Z3 = y * z3
    fe_mul(B, s2p, S1);
    fe_dbl(B, B);                    // (S2 - S1)^2 = c s2p^2 + S1^2 - y * B
    exact = exact || fe_is_zero(B);
    fe_sqr(t, s2p);
    fe_mul(A, c, t);
    fe_sqr(t, S1);
    fe_add(A, A, t);
    fe_sqr(HH, H);
    fe_mul(K, H, HH);                // H^3
    fe_sub(A, A, K);
    fe_mul(V, U1, HH);
    fe_sub(A, A, V);
    fe_sub(A, A, V);                 // - 2 U1 H^2 :  X3 = A - y B
    fe_sqr(t, z3);
    fe_mul(W0, c, t);                // Z3^2 = c z3^2
    fe_mul(t, rfe, W0);
    fe_sub(D, A, t);                 // X3 == r Z3^2  <=>  y B == D
    if (ext) {
        // Y3 = (y s2p - S1)(V - X3) - S1 H^3 = E + y F
        fe E, F;
        fe_mul(K, K, S1);            // K = S1 H^3
        fe_sub(V, V, A);             // V - A
        fe_mul(E, c, s2p);
        fe_mul(E, E, B);
        fe_mul(t, S1, V);
        fe_sub(E, E, t);
        fe_sub(E, E, K);             // E = c s2p B - S1 (V - A) - K
        fe_mul(F, s2p, V);
        fe_mul(t, S1, B);
        fe_sub(F, F, t);             // F = s2p (V - A) - S1 B
        fe_mul(E, E, B);
        fe_mul(F, F, D);
        fe_add(ext[0], E, F);        // N = E B + F D
        fe_mul(ext[1], W0, z3);      // CG = c z3^3
    }
    return exact;
}

// Curve side for one item.  Returns 0 (verdict 0 is final), SV_NS_PENDING (park filled) or SV_NS_EXACT.  `park` may alias w.
SV_HD u32 ecdsa33_nosqrt_curve_side(const sv_work* w, const u8* key33, const u8* sig64, const ge_mem* gtab, qtab_entry* tab,
                                    sv_ns_park* park, bool store, unsigned sync_threads = 0) {
    const u32 flags = w->flags;
    bool ok = (flags & SV_WF_VALID) != 0;
    const u8 pfx = key33[0];
    fe x, c, seven;
    ok = (pfx == 2 || pfx == 3) && ok;       // eckey_impl.h:17
    ok = fe_set_b32(x, key33 + 1) && ok;     // x < p  (group_impl.h:334 via fe_set_b32_limit)
    fe_set_u32(seven, 7);
    fe_sqr(c, x);
    fe_mul(c, c, x);
    fe_add(c, c, seven);
    {
        ge Qp;  // Q' = (c x, c^2) on E'
        fe_mul(Qp.x, c, x);
        fe_sqr(Qp.y, c);
        fe zc;
        qtable_build(tab, zc, Qp, sync_threads);
        gej S;
        ecmult_ladder_q(S, w, tab, zc, sync_threads);
        // the table is dead: park S' there while the comb runs
        fe_to_words(tab[0].x, S.x);
        fe_to_words(tab[0].y, S.y);
        fe_to_words(tab[0].h, S.z);
        tab[1].x[0] = S.inf;
    }
    gej T;
    T.inf = 1;
    fe_set_zero(T.x);
    fe_set_zero(T.y);
    fe_set_zero(T.z);
    ecmult_comb_add(T, w, gtab, sync_threads);
    bool exact = T.inf || tab[1].x[0] != 0 || (flags & SV_WF_R_PLUS_N) != 0;
    // c again (cheaper than keeping 8 registers alive across ladder and comb)
    fe_set_b32(x, key33 + 1);
    fe_sqr(c, x);
    fe_mul(c, c, x);
    fe_add(c, c, seven);
    fe X1, Y1, Zs, B, D, rfe;
    fe_from_words(X1, tab[0].x);
    fe_from_words(Y1, tab[0].y);
    fe_from_words(Zs, tab[0].h);
    fe_set_b32(rfe, sig64);          // r < n < p
    exact = ns_linear_form(D, B, X1, Y1, Zs, T, c, rfe) || exact;
    if (!ok) return 0u;
    if (exact) return SV_NS_EXACT;
    if (store) {
        fe_to_words(park->d, D);
        fe_to_words(park->b, B);
        fe_to_words(park->c, c);
    }
    return SV_NS_PENDING;
}

// verdicts for cnt (<= SV_FINAL_BATCH) consecutive items; verdict[i] holds the code ecdsa33_nosqrt_curve_side returned
// aux (optional, one byte per item): bit 0 = key decodes, bit 1 = signature encoding parsed — a valid signature proves its
// key; only for the others (rare in honest traffic) is the key decoded with the real square root.
SV_HD void ecdsa33_nosqrt_final_batch(u8* verdict, const sv_work* work, const u8* key33, const u8* sig64, const ge_mem* gtab,
                                      int cnt, u8* aux = nullptr) {
    fe pre[SV_FINAL_BATCH];
    fe acc, one;
    fe_set_u32(one, 1);
    for (int i = 0; i < cnt; i++) {
        const sv_ns_park* pk = reinterpret_cast<const sv_ns_park*>(work + i);
        fe b;
        fe_from_words(b, pk->b);
        if (verdict[i] != SV_NS_PENDING) b = one;
        if (i == 0) pre[0] = b; else fe_mul(pre[i], pre[i - 1], b);
    }
    fe_inv(acc, pre[cnt - 1]);
    // Items that need the real square root after all are only noted here and worked off in loops of their own below: the
    // lanes of a warp then run that (long) code side by side, whichever of their 16 items it concerns, instead of once per
    // loop index in which any lane needs it.
    u32 todo_key = 0, todo_exact = 0;
    for (int i = cnt - 1; i >= 0; i--) {
        const sv_ns_park* pk = reinterpret_cast<const sv_ns_park*>(work + i);
        const u32 code = verdict[i];
        fe b, bi;
        fe_from_words(b, pk->b);
        if (code != SV_NS_PENDING) b = one;
        if (i > 0) {
            fe_mul(bi, acc, pre[i - 1]);
            fe_mul(acc, acc, b);
        } else {
            bi = acc;
        }
        // the flags word of the work record lies past the parked D, B, c and is still intact
        const u32 parsed = (work[i].flags & SV_WF_PARSED) ? 2u : 0u;
        if (code == SV_NS_PENDING) {
            fe d, c, y, yy;
            fe_from_words(d, pk->d);
            fe_from_words(c, pk->c);
            fe_mul(y, d, bi);
            fe_normalize(y);
            fe_sqr(yy, y);
            bool good = fe_equal(yy, c) && (fe_is_odd(y) == (key33[33 * i] == 3));
            verdict[i] = good ? 1 : 0;
            if (aux) aux[i] = (u8)(1u | parsed);  // a valid signature proves its key
            if (!good) todo_key |= 1u << i;
        } else if (code == SV_NS_EXACT) {
            todo_exact |= 1u << i;
        } else {
            verdict[i] = 0;
            todo_key |= 1u << i;
        }
    }
    while (todo_exact) {
        int i = 0;
        while (!((todo_exact >> i) & 1u)) i++;
        todo_exact &= todo_exact - 1u;
        qtab_entry tab[8];
        bool kd;
        verdict[i] = (u8)verify_curve_side(SV_KIND_ECDSA33, work + i, key33 + 33 * i, sig64 + 64 * i, gtab, tab, &kd);
        if (aux) aux[i] = (u8)((kd ? 1u : 0u) | ((work[i].flags & SV_WF_PARSED) ? 2u : 0u));
    }
    while (aux && todo_key) {
        int i = 0;
        while (!((todo_key >> i) & 1u)) i++;
        todo_key &= todo_key - 1u;
        ge Q;
        bool kd = key_decode(Q, SV_KIND_ECDSA33, key33 + 33 * i);
        aux[i] = (u8)((kd ? 1u : 0u) | ((work[i].flags & SV_WF_PARSED) ? 2u : 0u));
    }
}

// ---- BIP-340 without the square root ---------------------------------------------------------------------------------
// Same idea for x-only keys: P = lift_x(px) is the point with the EVEN root y of c = px^3 + 7 (extrakeys/main_impl.h:32-38),
// R = s*G - e*P must be finite with even y and x(R) == r (schnorrsig/main_impl.h:255-264).  With S = -e*P = (X1, Y1, y Zs) and
// T = s*G the sum has  X3 = A - y B,  Y3 = E + y F,  Z3 = y z3  (y^2 = c folded in), so
//     x(R) == r   <=>  y = D / B,  D = A - r c z3^2          and then     y(R) = (E B + F D) / (D c z3^3).
// k_main parks D, B, N = E B + F D and CG = c z3^3; k_final_schnorr_ns inverts B * D * CG once per signature (batched) and
// checks  (D/B)^2 == c,  D/B even,  N / (D CG) even.  Configurations outside the linear form go to the plain path.
struct alignas(16) sv_ns_park_schnorr {
    u32 d[8], b[8], n[8], cg[8];
};

SV_HD u32 schnorr_nosqrt_curve_side(const sv_work* w, const u8* xonly32, const u8* sig64, const ge_mem* gtab, qtab_entry* tab,
                                    sv_ns_park_schnorr* park, bool store, unsigned sync_threads = 0) {
    const u32 flags = w->flags;
    bool ok = (flags & SV_WF_VALID) != 0;
    fe x, c, seven;
    ok = fe_set_b32(x, xonly32) && ok;  // px < p  (extrakeys/main_impl.h:32)
    fe_set_u32(seven, 7);
    fe_sqr(c, x);
    fe_mul(c, c, x);
    fe_add(c, c, seven);
    {
        ge Qp;
        fe_mul(Qp.x, c, x);
        fe_sqr(Qp.y, c);
        fe zc;
        qtable_build(tab, zc, Qp, sync_threads);
        gej S;
        ecmult_ladder_q(S, w, tab, zc, sync_threads);
        fe_to_words(tab[0].x, S.x);
        fe_to_words(tab[0].y, S.y);
        fe_to_words(tab[0].h, S.z);
        tab[1].x[0] = S.inf;
    }
    gej T;
    T.inf = 1;
    fe_set_zero(T.x);
    fe_set_zero(T.y);
    fe_set_zero(T.z);
    ecmult_comb_add(T, w, gtab, sync_threads);
    bool exact = T.inf || tab[1].x[0] != 0;
    fe_set_b32(x, xonly32);
    fe_sqr(c, x);
    fe_mul(c, c, x);
    fe_add(c, c, seven);
    fe X1, Y1, Zs, B, D, rfe, ext[2];
    fe_from_words(X1, tab[0].x);
    fe_from_words(Y1, tab[0].y);
    fe_from_words(Zs, tab[0].h);
    fe_set_b32(rfe, sig64);          // r < p checked by the scalar side (flags)
    exact = ns_linear_form(D, B, X1, Y1, Zs, T, c, rfe, ext) || exact;
    if (!ok) return 0u;
    if (exact) return SV_NS_EXACT;
    if (store) {
        fe_to_words(park->d, D);
        fe_to_words(park->b, B);
        fe_to_words(park->n, ext[0]);
        fe_to_words(park->cg, ext[1]);
    }
    return SV_NS_PENDING;
}

SV_HD void schnorr_nosqrt_final_batch(u8* verdict, const sv_work* work, const u8* xonly32, const u8* sig64, const ge_mem* gtab,
                                      int cnt) {
    fe pre[SV_FINAL_BATCH];
    fe acc, one;
    fe_set_u32(one, 1);
    for (int i = 0; i < cnt; i++) {
        const sv_ns_park_schnorr* pk = reinterpret_cast<const sv_ns_park_schnorr*>(work + i);
        fe v = one;
        if (verdict[i] == SV_NS_PENDING) {
            fe d, b, cg;
            fe_from_words(d, pk->d);
            fe_from_words(b, pk->b);
            fe_from_words(cg, pk->cg);
            fe_mul(v, d, cg);
            fe_mul(v, v, b);      // B * D * CG
            if (fe_is_zero(v)) v = one;  // D == 0 (B, CG are non-zero here): y would be 0, never a root of c != 0 -> rejected below
        }
        if (i == 0) pre[0] = v; else fe_mul(pre[i], pre[i - 1], v);
    }
    fe_inv(acc, pre[cnt - 1]);
    u32 todo_exact = 0;
    for (int i = cnt - 1; i >= 0; i--) {
        const sv_ns_park_schnorr* pk = reinterpret_cast<const sv_ns_park_schnorr*>(work + i);
        const u32 code = verdict[i];
        fe d, b, cg, w, v = one, vi;
        if (code == SV_NS_PENDING) {
            fe_from_words(d, pk->d);
            fe_from_words(b, pk->b);
            fe_from_words(cg, pk->cg);
            fe_mul(w, d, cg);     // W = D CG
            fe_mul(v, w, b);
            if (fe_is_zero(v)) v = one;
        }
        if (i > 0) {
            fe_mul(vi, acc, pre[i - 1]);
            fe_mul(acc, acc, v);
        } else {
            vi = acc;
        }
        if (code == SV_NS_PENDING) {
            fe x, c, seven, y, yy, yr, nn, t;
            fe_set_b32(x, xonly32 + 32 * i);
            fe_set_u32(seven, 7);
            fe_sqr(c, x);
            fe_mul(c, c, x);
            fe_add(c, c, seven);
            fe_mul(t, w, vi);     // 1 / B
            fe_mul(y, d, t);      // y = D / B
            fe_normalize(y);
            fe_sqr(yy, y);
            fe_mul(t, b, vi);     // 1 / W
            fe_from_words(nn, pk->n);
            fe_mul(yr, nn, t);    // y(R) = N / W
            fe_normalize(yr);
            bool good = !fe_is_zero(d) && fe_equal(yy, c) && !fe_is_odd(y) && !fe_is_odd(yr);
            verdict[i] = good ? 1 : 0;
        } else if (code == SV_NS_EXACT) {
            todo_exact |= 1u << i;
        } else {
            verdict[i] = 0;
        }
    }
    while (todo_exact) {  // a loop of its own: see ecdsa33_nosqrt_final_batch
        int i = 0;
        while (!((todo_exact >> i) & 1u)) i++;
        todo_exact &= todo_exact - 1u;
        qtab_entry tab[8];
        verdict[i] = (u8)verify_curve_side(SV_KIND_SCHNORR, work + i, xonly32 + 32 * i, sig64 + 64 * i, gtab, tab);
    }
}

// k*G (k != 0) as a normalised affine point through the fixed-base comb alone (signer of the synthetic workload generator,
// ecmult KAT of the self test).  Not constant time.
SV_HD void ecmult_gen_comb(ge& out, const sc& k, const ge_mem* gtab) {
    sv_work w;
    sc_prepare_u1(w, k);
    gej R;
    R.inf = 1;
    fe_set_zero(R.x); fe_set_zero(R.y); fe_set_zero(R.z);
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
    for (int row = 0; row < 16; row++) {
        int d = w.gd[row];
        if (d != 0) {
            ge p;
            u32 a = (u32)(d < 0 ? -d : d);
            ge_from_mem(p, gtab + (size_t)row * SV_GT_ROW + (a - 1));
            if (d < 0) fe_neg(p.y, p.y);
            gej_add_ge(R, R, p);
        }
    }
    fe zi;
    fe_inv(zi, R.z);
    ge_set_gej_zinv(out, R, zi);
    fe_normalize(out.x);
    fe_normalize(out.y);
}

// =================================================================================================
// small-batch path: ONE verification spread over three cooperating warps (k_small, engine.cu)
// =================================================================================================
// A lone verification on the throughput kernels is a single dependent chain of ~2,000 field operations plus a Fermat
// inversion, ~1.1 ms however few signatures there are (profiles/r2_latency_before_small_path.json).  The independent
// pieces of R = u1*G + k1*Q + k2*(lambda*Q) are therefore given to different warps of one CTA (different SM
// sub-partitions, so each has a multiplier pipe of its own), lane l of every warp working on item l of the CTA:
//   phase A   warp 0: key decode + odd-multiples table of Q        | warp 1: scalar side (s^-1, u1, u2, GLV, recoding)
//   phase B   warp 0: half ladder k1*Q  | warp 1: half ladder k2*(lambda*Q)  | warp 2: comb sum u1*G
//   phase C   warp 0: R = (R1 + R2) + u1*G with full Jacobian additions, final comparison
// The accept/reject rules are the same functions the throughput path uses (ecdsa_parse, ecdsa_finish_prep, schnorr_prep,
// key_decode, ecdsa_final, schnorr_final); only the schedule of the group operations differs.
struct alignas(16) sv_small_item {
    qtab_entry tab[8];  // effective-affine odd multiples of Q (x, y, beta*x)
    u32 zc[8];          // their common Z
    sv_work w;
    sv_jac r1, r2, p3;  // partial sums (r1, r2 on the scaled curve, p3 in true coordinates)
    u32 key_ok, pad[3];
};

SV_HD void small_key_side(int kind, const u8* key, sv_small_item* it) {
    ge Q;
    it->key_ok = key_decode(Q, kind, key) ? 1u : 0u;
    fe zc;
    qtable_build(it->tab, zc, Q);
    fe_to_words(it->zc, zc);
}
// scalar side of ONE signature: what k_prep_inv + k_prep_finish / k_prep_schnorr compute, without batching
SV_HD void small_scalar_side(int kind, const u8* msg32, const u8* key, const u8* sig64, sv_small_item* it) {
    if (kind == SV_KIND_SCHNORR) {
        schnorr_prep(it->w, sig64, key, msg32);
        return;
    }
    sc r, s, m, sinv;
    bool parsed = false;
    bool ok = ecdsa_parse(r, s, m, sig64, msg32, &parsed);
    if (!ok) {
        SV_UNROLL
        for (int k = 0; k < 8; k++) s.v[k] = (k == 0);
    }
    sc_inverse_var(sinv, s);
    ecdsa_finish_prep(it->w, ok, r, m, sinv, parsed);
}
// one GLV half: R = (+-|k|) * Q (or lambda*Q) on the scaled curve, 33 regular signed-odd-digit windows
SV_HD void ecmult_half_ladder(gej& R, const u32* mag, bool lam, const qtab_entry* tab) {
    u32 t = mag[4];
    u32 sgn = t >> 31;
    ge p;
    qtable_fetch(p, tab, ((t >> 1) & 7u) + 8u, sgn, lam);  // top window: digit 2*(mag >> 129) + 1, always positive
    gej_set_ge(R, p);
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
    for (int i = 31; i >= 0; i--) {
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
        for (int j = 0; j < 4; j++) gej_double(R, R);
        qtable_fetch(p, tab, window4(mag, i), sgn, lam);
        gej_add_ge(R, R, p);
    }
}
SV_HD void small_jac_store(sv_jac* out, const gej& R) {
    fe_to_words(out->x, R.x);
    fe_to_words(out->y, R.y);
    fe_to_words(out->z, R.z);
    out->inf = R.inf;
    out->ok = 1;
}
SV_HD void small_jac_load(gej& R, const sv_jac* in) {
    fe_from_words(R.x, in->x);
    fe_from_words(R.y, in->y);
    fe_from_words(R.z, in->z);
    R.inf = in->inf;
}
SV_HD void small_half_ladder(sv_small_item* it, int half) {
    gej R;
    ecmult_half_ladder(R, half ? it->w.k2 : it->w.k1, half != 0, it->tab);
    small_jac_store(half ? &it->r2 : &it->r1, R);
}
// u1*G as a Jacobian sum of the 16 comb points (infinity for u1 == 0)
SV_HD void small_comb(sv_small_item* it, const ge_mem* gtab) {
    gej R;
    R.inf = 1;
    fe_set_zero(R.x);
    fe_set_zero(R.y);
    fe_set_zero(R.z);
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
    for (int row = 0; row < 16; row++) {
        int d = it->w.gd[row];
        if (d != 0) {
            ge p;
            u32 a = (u32)(d < 0 ? -d : d);
            ge_from_mem(p, gtab + (size_t)row * SV_GT_ROW + (a - 1));
            if (d < 0) fe_neg(p.y, p.y);
            gej_add_ge(R, R, p);
        }
    }
    small_jac_store(&it->p3, R);
}
SV_HD u32 small_finish(int kind, sv_small_item* it, const u8* sig64, bool* key_ok = nullptr) {
    gej R, T;
    small_jac_load(R, &it->r1);
    small_jac_load(T, &it->r2);
    gej_add_gej(R, R, T);  // on the scaled curve: the formulas never use the curve constant
    fe zc;
    fe_from_words(zc, it->zc);
    fe_mul(R.z, R.z, zc);  // back to true coordinates
    small_jac_load(T, &it->p3);
    gej_add_gej(R, R, T);
    u32 flags = it->w.flags;
    bool ok = (flags & SV_WF_VALID) != 0 && it->key_ok != 0;
    if (key_ok) *key_ok = it->key_ok != 0;
    u32 v = (kind == SV_KIND_SCHNORR) ? schnorr_final(R, sig64, true) : ecdsa_final(R, sig64, flags);
    return ok ? v : 0u;
}
// ---- small-batch path without the square root (see "without the square root" above) ---------------------------------
// Written for both key kinds; the engine uses it for BIP-340 only (k_small<SCHNORR, true>) — for compressed-key ECDSA the one
// division per signature costs what the square root cost (measured, engine.cu launch_small), so kind 0 keeps the plain flow
// in the small-batch kernel.  The host build tests both.
// phase A builds the table of Q' = (c x, c^2) on the isomorphic curve, the half ladders and the comb run unchanged, and the
// finish assembles the linear form from S' = R1 + R2 and T and settles it with one field inversion per signature (no batch
// to share it with here).  key_ok then only says "the key's encoding is acceptable"; whether x is on the curve comes out of
// the final comparison.  Configurations the linear form does not cover are verified by the plain sequential path.
SV_HD void small_key_side_ns(int kind, const u8* key, sv_small_item* it) {
    fe x, c, seven;
    bool ok;
    if (kind == SV_KIND_ECDSA33) {
        const u8 pfx = key[0];
        ok = (pfx == 2 || pfx == 3);            // eckey_impl.h:17
        ok = fe_set_b32(x, key + 1) && ok;
    } else {
        ok = fe_set_b32(x, key);                // extrakeys/main_impl.h:32
    }
    it->key_ok = ok ? 1u : 0u;
    fe_set_u32(seven, 7);
    fe_sqr(c, x);
    fe_mul(c, c, x);
    fe_add(c, c, seven);
    ge Qp;
    fe_mul(Qp.x, c, x);
    fe_sqr(Qp.y, c);
    fe zc;
    qtable_build(it->tab, zc, Qp);
    fe_to_words(it->zc, zc);
}

// key_ok (optional): whether the key decodes (secp256k1_ec_pubkey_parse / xonly_pubkey_parse would accept it)
SV_HD u32 small_finish_ns(int kind, sv_small_item* it, const u8* key, const u8* sig64, const ge_mem* gtab, bool* key_ok = nullptr) {
    const u32 flags = it->w.flags;
    const bool ok = (flags & SV_WF_VALID) != 0 && it->key_ok != 0;
    gej S, T;
    small_jac_load(S, &it->r1);
    small_jac_load(T, &it->r2);
    gej_add_gej(S, S, T);   // on the isomorphic, scaled curve: the formulas never use the curve constant
    fe zc;
    fe_from_words(zc, it->zc);
    fe_mul(S.z, S.z, zc);
    small_jac_load(T, &it->p3);
    bool exact = S.inf || T.inf || (kind == SV_KIND_ECDSA33 && (flags & SV_WF_R_PLUS_N) != 0);
    fe x, c, seven, rfe, D, B, ext[2];
    fe_set_b32(x, kind == SV_KIND_ECDSA33 ? key + 1 : key);
    fe_set_u32(seven, 7);
    fe_sqr(c, x);
    fe_mul(c, c, x);
    fe_add(c, c, seven);
    fe_set_b32(rfe, sig64);
    exact = ns_linear_form(D, B, S.x, S.y, S.z, T, c, rfe, kind == SV_KIND_SCHNORR ? ext : nullptr) || exact;
    u32 v = 0;
    bool kd = false, kd_known = false;
    if (ok && exact) {
        // rare (a signer steering the scalars): the plain path, one thread
        v = verify_curve_side(kind, &it->w, key, sig64, gtab, it->tab, &kd);
        kd_known = true;
    } else if (ok) {
        fe inv, y, yy, t;
        if (kind == SV_KIND_SCHNORR) {
            fe w;
            fe_mul(w, D, ext[1]);          // W = D CG
            fe_mul(t, w, B);
            bool zero = fe_is_zero(t);     // D == 0: y would be 0, never a root of c != 0
            if (zero) fe_set_u32(t, 1);
            fe_inv_var(inv, t);            // 1 / (B W)
            fe_mul(t, w, inv);             // 1 / B
            fe_mul(y, D, t);
            fe_normalize(y);
            fe_sqr(yy, y);
            fe yr;
            fe_mul(t, B, inv);             // 1 / W
            fe_mul(yr, ext[0], t);         // y(R) = N / W
            fe_normalize(yr);
            v = (!zero && fe_equal(yy, c) && !fe_is_odd(y) && !fe_is_odd(yr)) ? 1u : 0u;   // main_impl.h:255-264
        } else {
            fe_inv_var(inv, B);
            fe_mul(y, D, inv);
            fe_normalize(y);
            fe_sqr(yy, y);
            v = (fe_equal(yy, c) && (fe_is_odd(y) == (key[0] == 3))) ? 1u : 0u;
        }
        if (v) { kd = true; kd_known = true; }
    }
    if (key_ok) {
        if (!kd_known) {
            ge Q;
            kd = key_decode(Q, kind, key);
        }
        *key_ok = kd;
    }
    return v;
}

// ---- half ladder on a PAIR of lanes -------------------------------------------------------------------------------
// A half ladder is one dependent chain of 128 doublings and 33 additions: 1,259 field multiplications one after another
// set the latency of a lone verification.  Inside one doubling / addition, however, several multiplications are independent
// of each other; two neighbouring lanes (2k, 2k+1) of a warp therefore share one half ladder: each step both lanes multiply
// (different operands), results they need from each other cross with warp shuffles.  A doubling takes 4 multiplication
// steps instead of 7, a mixed addition 6 instead of 11.  Both lanes hold the full point before and after every operation.
// The case analysis is that of gej_double / gej_add_ge.
struct pair_lane {
    int role;  // 0 / 1 inside the pair
#if !SV_DEVICE_CODE
    struct pair_mailbox* mb;  // host build: the two lanes are two threads meeting at a mailbox (tests/host_emul)
#endif
};
#if SV_DEVICE_CODE
SV_HD void pair_swap(const pair_lane&, fe& recv, const fe& send) {
    unsigned m = __activemask();  // both lanes of a pair always take the same branches
    SV_UNROLL
    for (int i = 0; i < 8; i++) recv.v[i] = __shfl_xor_sync(m, send.v[i], 1);
}
#else
SV_HD void pair_swap(const pair_lane& L, fe& recv, const fe& send);  // tests/host_emul/emul.cpp
#endif
SV_HD void fe_sel(fe& r, bool c, const fe& a, const fe& b) {  // r = c ? a : b
    SV_UNROLL
    for (int i = 0; i < 8; i++) r.v[i] = c ? a.v[i] : b.v[i];
}

// R = 2R.  steps: [A = X^2 | B = Y^2]  [T = Y*Z | C = B^2]  [S = (X+B)^2 | EE = (3A)^2]  [ - | M = E*(D - X3)]
SV_HD void pair_double(const pair_lane& L, gej& R) {
    const bool r1 = L.role != 0;
    fe a, b, t, u, o1, o2;
    fe_sel(t, r1, R.y, R.x);
    fe_sqr(a, t);                       // lane0: A          lane1: B
    fe_sel(o1, r1, a, R.y);
    fe_sel(o2, r1, a, R.z);
    fe_mul(b, o1, o2);                  // lane0: T = Y*Z    lane1: C = B^2
    pair_swap(L, t, a);                 // lane0 gets B      lane1 gets A
    fe e;
    fe_mul3(e, r1 ? t : a);             // E = 3A (meaningful on lane 1; lane 0 computes it too: it holds A in `a`)
    fe_add(u, R.x, r1 ? a : t);         // X + B
    fe_sel(o1, r1, e, u);
    fe s;
    fe_sqr(s, o1);                      // lane0: S = (X+B)^2   lane1: EE = E^2
    fe A_, C_;
    fe_sel(A_, r1, t, a);               // A on both lanes
    pair_swap(L, u, r1 ? b : s);        // lane0 sends S, lane1 sends C:  lane0 gets C, lane1 gets S
    fe S_;
    fe_sel(S_, r1, u, s);
    fe_sel(C_, r1, b, u);
    fe d;
    fe_sub(d, S_, A_);
    fe_sub(d, d, C_);
    fe_dbl(d, d);                       // D on both lanes
    fe x3, m, c8, z3;
    fe_sub(x3, s, d);                   // lane1: X3 = EE - 2D (lane 0: garbage)
    fe_sub(x3, x3, d);
    fe_sub(t, d, x3);
    fe_mul(m, e, t);                    // lane1: M = E*(D - X3)
    fe_mul8(c8, C_);
    fe y3;
    fe_sub(y3, m, c8);                  // lane1: Y3
    fe_dbl(z3, b);                      // lane0: Z3 = 2T
    pair_swap(L, t, r1 ? x3 : z3);      // lane0 gets X3, lane1 gets Z3
    pair_swap(L, u, y3);                // lane0 gets Y3
    fe_sel(R.x, r1, x3, t);
    fe_sel(R.y, r1, y3, u);
    fe_sel(R.z, r1, t, z3);
}

// R = R + p (p affine).  steps: [zz = Z^2 | -] [u2 = px*zz | zzz = Z*zz] [hh = h^2 | s2 = py*zzz] [hhh = h*hh | rr^2]
//                              [v = X*hh | Z3 = Z*h] [rr*(v - X3) | hhh*Y]
SV_HD void pair_add_ge(const pair_lane& L, gej& R, const ge& p) {
    const bool r1 = L.role != 0;
    if (R.inf) {
        gej_set_ge(R, p);
        return;
    }
    fe zz, t, u, w, h, rr, o1, o2;
    fe_sqr(zz, R.z);                    // both lanes (same operand): zz
    fe_sel(o1, r1, R.z, p.x);
    fe_mul(t, o1, zz);                  // lane0: u2 = px*zz     lane1: zzz = Z*zz
    fe_sub(h, t, R.x);                  // lane0: h
    fe_sel(o1, r1, p.y, h);
    fe_sel(o2, r1, t, h);
    fe_mul(u, o1, o2);                  // lane0: hh = h^2       lane1: s2 = py*zzz
    fe_sub(rr, u, R.y);                 // lane1: rr
    pair_swap(L, w, r1 ? rr : h);       // lane0 gets rr, lane1 gets h
    fe H_, RR_;
    fe_sel(H_, r1, w, h);
    fe_sel(RR_, r1, rr, w);
    if (fe_is_zero(H_)) {               // same x: double or cancel (group_impl.h:595-605); both lanes agree on the branch
        if (fe_is_zero(RR_)) pair_double(L, R);
        else {
            R.inf = 1;
            fe_set_zero(R.x); fe_set_zero(R.y); fe_set_zero(R.z);
        }
        return;
    }
    fe_sel(o1, r1, RR_, H_);
    fe_sel(o2, r1, RR_, u);
    fe q;
    fe_mul(q, o1, o2);                  // lane0: hhh = h*hh     lane1: rr2 = rr^2
    fe_sel(o1, r1, R.z, R.x);
    fe_sel(o2, r1, H_, u);
    fe g;
    fe_mul(g, o1, o2);                  // lane0: v = X*hh       lane1: Z3 = Z*h
    pair_swap(L, w, q);                 // lane0 gets rr2, lane1 gets hhh
    fe x3;
    fe_sub(x3, w, q);                   // lane0: rr2 - hhh
    fe_sub(x3, x3, g);
    fe_sub(x3, x3, g);                  // lane0: X3 = rr2 - hhh - 2v
    fe_sub(t, g, x3);                   // lane0: v - X3
    fe_sel(o1, r1, w, RR_);
    fe_sel(o2, r1, R.y, t);
    fe m;
    fe_mul(m, o1, o2);                  // lane0: rr*(v - X3)    lane1: hhh*Y
    pair_swap(L, t, m);                 // lane0 gets hhh*Y
    fe y3;
    fe_sub(y3, m, t);                   // lane0: Y3
    pair_swap(L, w, r1 ? g : x3);       // lane0 gets Z3, lane1 gets X3
    pair_swap(L, u, y3);                // lane1 gets Y3
    fe_sel(R.x, r1, w, x3);
    fe_sel(R.y, r1, u, y3);
    fe_sel(R.z, r1, g, w);
    R.inf = 0;
}
SV_HD void ecmult_half_ladder_pair(const pair_lane& L, gej& R, const u32* mag, bool lam, const qtab_entry* tab) {
    u32 t = mag[4];
    u32 sgn = t >> 31;
    ge p;
    qtable_fetch(p, tab, ((t >> 1) & 7u) + 8u, sgn, lam);
    gej_set_ge(R, p);
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
    for (int i = 31; i >= 0; i--) {
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
        for (int j = 0; j < 4; j++) pair_double(L, R);
        qtable_fetch(p, tab, window4(mag, i), sgn, lam);
        pair_add_ge(L, R, p);
    }
}
SV_HD void small_half_ladder_pair(const pair_lane& L, sv_small_item* it, int half) {
    gej R;
    ecmult_half_ladder_pair(L, R, half ? it->w.k2 : it->w.k1, half != 0, it->tab);
    if (L.role == 0) small_jac_store(half ? &it->r2 : &it->r1, R);
}

// ---- recovery on the small-batch path: warp 0 lifts R and builds its table in place of the key side, warp 1 runs the
// scalar side with a lone inversion of r, the half ladders and the comb are unchanged, and the finish leaves Jacobian
// coordinates with one field inversion per item (no batch to share it with here)
SV_HD void small_recover_key_side(const u8* sig64, u32 recid, sv_small_item* it) {
    ge R;
    it->key_ok = recover_lift(R, sig64, recid) ? 1u : 0u;
    fe zc;
    qtable_build(it->tab, zc, R);
    fe_to_words(it->zc, zc);
}
SV_HD void small_recover_scalar_side(const u8* msg32, const u8* sig64, u32 recid, sv_small_item* it) {
    sc r, s, m, rinv, d;
    bool ok, parsed;
    recover_parse(r, s, m, ok, parsed, sig64, msg32, recid);
    d = r;
    if (!ok) {
        SV_UNROLL
        for (int k = 0; k < 8; k++) d.v[k] = (k == 0);
    }
    sc_inverse_var(rinv, d);
    recover_finish_prep(it->w, ok, parsed, r, s, m, rinv);
}
SV_HD void small_recover_finish(sv_small_item* it, u32 recid, u8* xy64, u8* status) {
    gej R, T;
    small_jac_load(R, &it->r1);
    small_jac_load(T, &it->r2);
    gej_add_gej(R, R, T);  // on the scaled curve
    fe zc;
    fe_from_words(zc, it->zc);
    fe_mul(R.z, R.z, zc);
    small_jac_load(T, &it->p3);
    gej_add_gej(R, R, T);
    const u32 flags = it->w.flags;
    const bool usable = recover_lift_allowed(flags, recid) && it->key_ok != 0 && !R.inf;
    ge a;
    if (usable) {
        fe zi;
        fe_inv_var(zi, R.z);
        ge_set_gej_zinv(a, R, zi);
    }
    recover_emit(xy64, status, usable ? &a : nullptr, (flags & SV_WF_PARSED) != 0);
}

// the three phases run one after another (host build of the kernel source, tests/host_emul)
SV_HD u32 verify_small_sequential(int kind, const u8* msg32, const u8* key, const u8* sig64, const ge_mem* gtab,
                                  sv_small_item* it, bool nosqrt = false) {
    nosqrt = nosqrt && kind != SV_KIND_ECDSA_XY;
    if (nosqrt) small_key_side_ns(kind, key, it); else small_key_side(kind, key, it);
    small_scalar_side(kind, msg32, key, sig64, it);
    small_half_ladder(it, 0);
    small_half_ladder(it, 1);
    small_comb(it, gtab);
    return nosqrt ? small_finish_ns(kind, it, key, sig64, gtab) : small_finish(kind, it, sig64);
}

// =================================================================================================
// fixed-base table construction (K4)
// =================================================================================================

// bases[i] = 2^(16 i) * G, i = 0..15 (one thread)
SV_HD void gtable_make_bases(ge_mem* bases) {
    ge g;
    SV_UNROLL
    for (int i = 0; i < 8; i++) { g.x.v[i] = GE_GX[i]; g.y.v[i] = GE_GY[i]; }
    for (int i = 0; i < 16; i++) {
        ge_to_mem(&bases[i], g);
        gej j;
        gej_set_ge(j, g);
        for (int k = 0; k < 16; k++) gej_double(j, j);
        fe zi;
        fe_inv(zi, j.z);
        ge_set_gej_zinv(g, j, zi);
        fe_normalize(g.x);
        fe_normalize(g.y);
    }
}
// table entry e (0 <= e < SV_GT_ENTRIES): row = min(e / 32768, 15), d = e - row*32768 + 1; value d * bases[row]
SV_HD void gtable_make_entry(ge_mem* table, const ge_mem* bases, u32 e) {
    u32 row = e / SV_GT_ROW;
    if (row > 15) row = 15;
    u32 d = e - row * SV_GT_ROW + 1;  // 1 .. 65536
    ge b;
    ge_from_mem(b, &bases[row]);
    gej acc;
    acc.inf = 1;
    fe_set_zero(acc.x);
    fe_set_zero(acc.y);
    fe_set_zero(acc.z);
#if SV_DEVICE_CODE
#pragma unroll 1
#endif
    for (int bit = 16; bit >= 0; bit--) {
        if (!acc.inf) gej_double(acc, acc);
        if ((d >> bit) & 1u) gej_add_ge(acc, acc, b);
    }
    fe zi;
    ge a;
    fe_inv(zi, acc.z);
    ge_set_gej_zinv(a, acc, zi);
    fe_normalize(a.x);
    fe_normalize(a.y);
    ge_to_mem(&table[e], a);
}
