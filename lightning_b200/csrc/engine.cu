// engine.cu — kernels and C ABI of libcln_sigverify.so (sm_100a).
//
// Kernels (SURVEY.md §2.3 naming):
//   K4  k_gtable_bases / k_gtable_fill   fixed-base comb table d * 2^(16 i) * G, built once per context
//   K3  k_sha256d                        SHA-256d of message spans (gossip tails, BIP143 preimages)
//   K1a k_prep_inv + k_prep_finish       scalar side of ECDSA (32 signatures per thread share one s^-1 exponentiation;
//                                        then one thread per signature: u1, u2, GLV split, recoding)
//   K2a k_prep_schnorr                   scalar side of BIP-340 (tagged challenge hash, -e, recoding)
//   K1b/K2b k_main<kind>                 curve side: thread per verification, persistent grid.  kind 3 / 4 = compressed /
//                                        x-only keys WITHOUT the square root (verify.cuh): the default for kinds 0 / 2
//       k_final_ecdsa33, k_final_schnorr_ns   batched division that settles the parked linear conditions of kinds 3 / 4
//       k_final_schnorr                  plain BIP-340 flow: affine R from the parked Jacobian R (batched inversion)
//       k_small<kind>                    one-launch latency path for small batches (5 warps per 32 verifications)
//       k_prep_recover_*, k_main<5>, k_final_recover, k_small<5>   public-key recovery (sv_recover_host)
//       k_main_shared, k_dedup_*, k_sharedkey_build_many   one multiples table per distinct key (same-key / gossip batches)
//       k_gossip_slice / _status, k_bip143, k_mixed_*       callers' data formats on the device (rows N1, N2, C3)
//       k_sb_* (batch.cu)                BIP-340 batch verification by random linear combination
//       k_pack_bitmap                    verdict bytes -> 1 bit per verification (ballot)
//       k_pubkey_parse                   batched pubkey_from_der
//       k_synth                          synthetic signed workload generator (benchmarks/tests)
//       k_probe_*                        integer-pipe microbenchmarks (roofline denominator)
//
// There is no host implementation of any of the arithmetic in this library: every entry point either
// runs the kernels or fails with an error code.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/cln_sigverify.h"
#include "verify.cuh"
#include "selftest.cuh"
#include "batch.cuh"  // constants and the host-testable stages; the kernels themselves are in batch.cu

// Build variants of the curve-side kernel (measured on B200, 1 M ECDSA33 verifications, profiles/):
//   default  SV_FE_INLINE + SV_MAIN_SYNC, 256 threads x 2 CTAs/SM : field arithmetic inlined, the warps of a CTA
//            re-converge at a __syncthreads() before every point operation so that they walk the (large) code
//            together and share instruction fetches                                    -> 43.7 M verifies/s
//   -DSV_NO_SYNC_INLINE  fe_mul/fe_sqr as real functions, 128 x 4, no barriers        -> 39.2 M verifies/s
//   (everything inlined WITHOUT barriers starves on instruction fetch                  -> 25.9 M verifies/s)
#if !defined(SV_NO_SYNC_INLINE) && !defined(SV_FE_INLINE)
#error "compile with -DSV_FE_INLINE -DSV_MAIN_SYNC (default build) or -DSV_NO_SYNC_INLINE; see lightning_b200/build.py"
#endif
#ifndef SV_MAIN_BLOCK
#ifdef SV_MAIN_SYNC
#define SV_MAIN_BLOCK 256
#else
#define SV_MAIN_BLOCK 128
#endif
#endif
#ifndef SV_MAIN_MINB
#define SV_MAIN_MINB (512 / SV_MAIN_BLOCK)
#endif
#ifdef SV_COMB_SMEM
#define SV_MAIN_SMEM (17 * 128 * 64)  // the variant's shared-memory comb table
#else
#define SV_MAIN_SMEM 0
#endif

// -------------------------------------------------------------------------------------------------
// kernels
// -------------------------------------------------------------------------------------------------
__global__ void k_gtable_bases(ge_mem* bases) {
    if (blockIdx.x == 0 && threadIdx.x == 0) gtable_make_bases(bases);
}
__global__ void __launch_bounds__(128) k_gtable_fill(ge_mem* table, const ge_mem* bases) {
    u32 e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < SV_GT_ENTRIES) gtable_make_entry(table, bases, e);
}

__global__ void __launch_bounds__(128) k_sha256d(const u8* data, const u64* off, const u32* len, size_t n, u8* out32) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sha256d_bytes(out32 + 32 * i, data + off[i], len[i]);
}

// scalar side, ECDSA, in two kernels.
//   k_prep_inv    : each thread owns SV_PREP_BATCH (32) consecutive signatures: range checks and ONE Fermat
//                   exponentiation mod n amortised by Montgomery's trick (3 mults + 1/32 of ~330 per signature).  Few
//                   threads, long serial chains: latency bound, so it does nothing else.  Leaves s^-1 and the check
//                   flags in the (not yet used) work record.
//   k_prep_finish : one thread per signature: u1 = m/s, u2 = r/s, GLV split, window recoding -> work record.
__global__ void __launch_bounds__(64) k_prep_inv(const u8* msg, const u8* sig, size_t n, sv_work* work) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t base = t * SV_PREP_BATCH;
    if (base >= n) return;
    int cnt = (int)((n - base < SV_PREP_BATCH) ? (n - base) : SV_PREP_BATCH);
    sc sv[SV_PREP_BATCH];
    u32 okmask = 0, parsedmask = 0;
#pragma unroll 1
    for (int j = 0; j < SV_PREP_BATCH; j++) {
        sc r, s, m;
        bool ok = false, parsed = false;
        if (j < cnt) ok = ecdsa_parse(r, s, m, sig + 64 * (base + j), msg + 32 * (base + j), &parsed);
        parsedmask |= (parsed ? 1u : 0u) << j;
        if (!ok) {
#pragma unroll
            for (int k = 0; k < 8; k++) s.v[k] = (k == 0);
        }
        okmask |= (ok ? 1u : 0u) << j;
        sv[j] = s;
    }
    sc_batch_inverse(sv, SV_PREP_BATCH);
#pragma unroll 1
    for (int j = 0; j < cnt; j++) {
        u32* w = reinterpret_cast<u32*>(work + base + j);
        fe_to_words(w, *reinterpret_cast<const fe*>(&sv[j]));  // words 0..7: s^-1
        w[8] = ((okmask >> j) & 1u) | (((parsedmask >> j) & 1u) << 1);
    }
}
__global__ void __launch_bounds__(128) k_prep_finish(const u8* msg, const u8* sig, size_t n, sv_work* work) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u32* wi = reinterpret_cast<const u32*>(work + i);
    sc sinv;
    fe tmp;
    fe_from_words(tmp, wi);
#pragma unroll
    for (int k = 0; k < 8; k++) sinv.v[k] = tmp.v[k];
    u32 f = wi[8];
    sc r, s, m;
    (void)ecdsa_parse(r, s, m, sig + 64 * i, msg + 32 * i);
    sv_work w;
    ecdsa_finish_prep(w, (f & 1u) != 0, r, m, sinv, (f & 2u) != 0);
    work[i] = w;
}

// scalar side of public-key recovery, split as for ECDSA: here r is the scalar to invert (recid in a byte array of its own)
__global__ void __launch_bounds__(64) k_prep_recover_inv(const u8* msg, const u8* sig, const u8* recid, size_t n, sv_work* work) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t base = t * SV_PREP_BATCH;
    if (base >= n) return;
    int cnt = (int)((n - base < SV_PREP_BATCH) ? (n - base) : SV_PREP_BATCH);
    sc rv[SV_PREP_BATCH];
    u32 okmask = 0, parsedmask = 0;
#pragma unroll 1
    for (int j = 0; j < SV_PREP_BATCH; j++) {
        sc r, s, m;
        bool ok = false, parsed = false;
        if (j < cnt) recover_parse(r, s, m, ok, parsed, sig + 64 * (base + j), msg + 32 * (base + j), recid[base + j]);
        parsedmask |= (parsed ? 1u : 0u) << j;
        if (!ok) {
#pragma unroll
            for (int k = 0; k < 8; k++) r.v[k] = (k == 0);
        }
        okmask |= (ok ? 1u : 0u) << j;
        rv[j] = r;
    }
    sc_batch_inverse(rv, SV_PREP_BATCH);
#pragma unroll 1
    for (int j = 0; j < cnt; j++) {
        u32* w = reinterpret_cast<u32*>(work + base + j);
        fe_to_words(w, *reinterpret_cast<const fe*>(&rv[j]));  // words 0..7: r^-1
        w[8] = ((okmask >> j) & 1u) | (((parsedmask >> j) & 1u) << 1);
    }
}
__global__ void __launch_bounds__(128) k_prep_recover_finish(const u8* msg, const u8* sig, const u8* recid, size_t n,
                                                             sv_work* work) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u32* wi = reinterpret_cast<const u32*>(work + i);
    sc rinv;
    fe tmp;
    fe_from_words(tmp, wi);
#pragma unroll
    for (int k = 0; k < 8; k++) rinv.v[k] = tmp.v[k];
    u32 f = wi[8];
    sc r, s, m;
    bool ok, parsed;
    recover_parse(r, s, m, ok, parsed, sig + 64 * i, msg + 32 * i, recid[i]);
    sv_work w;
    recover_finish_prep(w, (f & 1u) != 0, (f & 2u) != 0, r, s, m, rinv);
    work[i] = w;
}

__global__ void __launch_bounds__(128) k_prep_schnorr(const u8* msg, const u8* key, const u8* sig, size_t n,
                                                      sv_work* work) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sv_work w;
    schnorr_prep(w, sig + 64 * i, key + 32 * i, msg + 32 * i);
    work[i] = w;
}

// curve side: one thread per verification, persistent grid-stride loop.  Per-thread odd-multiples
// table lives in an HBM/L2-resident scratch slab (768 B per thread, 64-byte entries read with LDG.128).
// record used by lanes past the end of the batch: harmless scalars (k1 = k2 = 1, u1 = 0), never valid.
// (They must not alias a live record: the BIP-340 path overwrites records with the parked R.)
__device__ sv_work g_idle_work = {{1, 0, 0, 0, 0}, {1, 0, 0, 0, 0}, {0}, 0, {0}};

#ifdef SV_COMB_SMEM
__device__ const ge_mem* g_t8;  // 17 x 128 entries d * 2^(8 i) * G in global memory, source of the per-CTA shared copy
__global__ void k_t8_fill(ge_mem* t8, const ge_mem* gtab) {
    u32 e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= 17 * 128) return;
    u32 row = e / 128, d = e % 128 + 1;  // d * 2^(8 row) G = (d << (8 (row & 1))) * 2^(16 (row / 2)) G
    t8[e] = gtab[(size_t)(row >> 1) * SV_GT_ROW + ((d << (8 * (row & 1))) - 1)];
}
#endif
template <int KIND>
__global__ void __launch_bounds__(SV_MAIN_BLOCK, SV_MAIN_MINB)
    k_main(sv_work* work, const u8* __restrict__ key, const u8* __restrict__ sig, size_t n,
           const ge_mem* __restrict__ gtab, qtab_entry* scratch, u8* __restrict__ verdict, u8* keyok) {
    const size_t keylen = (KIND == SV_KIND_ECDSA33 || KIND == SV_KIND_ECDSA33_NS) ? 33
                          : (KIND == SV_KIND_ECDSA_XY ? 64 : (KIND == SV_KIND_RECOVER ? 1 : 32));
#ifdef SV_COMB_SMEM
    // VARIANT: the 17 x 128-entry 8-bit comb (136 KiB) is staged in shared memory once per (persistent) CTA by ONE bulk
    // asynchronous copy (cp.async.bulk: the TMA engine, UBLKCP in SASS), completion signalled on an mbarrier
    {
        extern __shared__ __align__(16) unsigned char sv_smem_raw[];
        __shared__ __align__(8) unsigned long long sv_bar;
        const unsigned bytes = 17u * 128u * (unsigned)sizeof(ge_mem);
        unsigned bar = (unsigned)__cvta_generic_to_shared(&sv_bar), dst = (unsigned)__cvta_generic_to_shared(sv_smem_raw);
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(dst), "l"(g_t8), "r"(bytes), "r"(bar) : "memory");
        }
        unsigned done = 0;
        while (!done)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(done) : "r"(bar) : "memory");
    }
#endif
#ifndef SV_MAP_INTERLEAVED
    size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    qtab_entry* tab = scratch + tid * 8;
    // CTA-uniform trip count (lanes past the end redo dummy work and discard the result) so that every thread
    // reaches every SV_SYNC() of the barrier-synchronised build
    for (size_t base = (size_t)blockIdx.x * blockDim.x; base < n; base += stride) {
        size_t i = base + threadIdx.x;
        bool active = i < n;
        size_t j = active ? i : 0;
        const unsigned part = SV_MAIN_BLOCK;  // every thread of the CTA reaches every re-convergence barrier
#else
    // VARIANT (measured 1.3 % slower at 1 M, profiles/r1_variants.md): interleaved item mapping — in round k thread t of
    // CTA c takes item k*T + t*G + c, so a partial last round keeps the first warps of EVERY CTA busy, the idle warps
    // leave, and the re-convergence barrier counts only the warps taking part.
    const unsigned G = gridDim.x, B = blockDim.x;
    const size_t T = (size_t)G * B;
    qtab_entry* tab = scratch + ((size_t)blockIdx.x * B + threadIdx.x) * 8;
    const size_t r = (size_t)threadIdx.x * G + blockIdx.x;
    for (size_t base = 0; base < n; base += T) {
        const size_t rem = n - base;
        unsigned act = B;
        if (rem < T) act = (rem > blockIdx.x) ? (unsigned)(((rem - blockIdx.x + G - 1) / G) < B ? ((rem - blockIdx.x + G - 1) / G) : B) : 0u;
        const unsigned part = (act + 31u) & ~31u;  // whole warps
        __syncthreads();  // all warps are out of the previous round's counted barriers before the count may change
        if (threadIdx.x >= part) return;  // only possible in the last round
        const size_t i = base + r;
        const bool active = r < rem;
        const size_t j = active ? i : 0;
#endif
        const sv_work* w = active ? (work + i) : &g_idle_work;
        if (KIND == SV_KIND_ECDSA33_NS) {
            // compressed-key ECDSA without the square root: D, B, c parked in the work record, k_final_ecdsa33 decides
            u32 code = ecdsa33_nosqrt_curve_side(w, key + keylen * j, sig + 64 * j, gtab, tab,
                                                 reinterpret_cast<sv_ns_park*>(work + j), active, part);
            if (active) verdict[i] = (u8)code;
        } else if (KIND == SV_KIND_SCHNORR_NS) {
            u32 code = schnorr_nosqrt_curve_side(w, key + keylen * j, sig + 64 * j, gtab, tab,
                                                 reinterpret_cast<sv_ns_park_schnorr*>(work + j), active, part);
            if (active) verdict[i] = (u8)code;
        } else if (KIND == SV_KIND_SCHNORR) {
            // park R in the work record; k_final_schnorr turns it into a verdict (batched inversion)
            bool ok = (w->flags & SV_WF_VALID) != 0;
            ge Q;
            ok = key_decode(Q, KIND, key + keylen * j) && ok;
            gej R;
            ecmult_uniform(R, w, Q, gtab, tab, part);
            if (active) schnorr_park(reinterpret_cast<sv_jac*>(work + i), R, ok);
        } else if (KIND == SV_KIND_RECOVER) {
            // public-key recovery: the recid byte sits in the key slot; Q is parked in the work record and
            // k_final_recover turns it into an affine key (batched inversion)
            const u32 recid = key[j];
            const u32 flags = w->flags;
            ge R;
            bool ok = recover_lift(R, sig + 64 * j, recid) && recover_lift_allowed(flags, recid);
            gej Q;
            ecmult_uniform(Q, w, R, gtab, tab, part);
            if (active) recover_park(reinterpret_cast<sv_jac*>(work + i), Q, ok, (flags & SV_WF_PARSED) != 0);
        } else {
            bool kd;
            u32 v = verify_curve_side(KIND, w, key + keylen * j, sig + 64 * j, gtab, tab, &kd, part);
            if (active) {
                verdict[i] = (u8)v;
                // gossip ingest distinguishes "undecodable key" / "unparsable signature" (malformed message) from a bad signature
                if (keyok) keyok[i] = (u8)((kd ? 1u : 0u) | ((w->flags & SV_WF_PARSED) ? 2u : 0u));
            }
        }
    }
}

// ---- small-batch path (verify.cuh "small-batch path"): one CTA = 5 warps x up to 32 items.  The inputs may live in host-mapped pinned memory (zero-copy: the CTA pulls its items into shared memory
// with warp-coalesced loads) or in device memory.  aux (optional): bit 0 = key decoded, bit 1 = signature encoding parsed.
#define SV_SMALL_ITEMS 32
template <int KIND, bool NOSQRT>
__global__ void __launch_bounds__(160, 1)
    k_small(const u8* __restrict__ msg, const u8* __restrict__ key, const u8* __restrict__ sig, size_t n,
            const ge_mem* __restrict__ gtab, u8* __restrict__ verdict, u8* __restrict__ aux) {
    // SV_KIND_RECOVER: the key slot holds the recid byte, verdict receives the status bytes and aux the 64-byte keys
    constexpr int keylen = (KIND == SV_KIND_ECDSA33) ? 33 : (KIND == SV_KIND_ECDSA_XY ? 64 : (KIND == SV_KIND_RECOVER ? 1 : 32));
    __shared__ sv_small_item items[SV_SMALL_ITEMS];
    __shared__ __align__(16) u8 in_msg[SV_SMALL_ITEMS * 32];
    __shared__ __align__(16) u8 in_key[SV_SMALL_ITEMS * 64];
    __shared__ __align__(16) u8 in_sig[SV_SMALL_ITEMS * 64];
    const size_t base = (size_t)blockIdx.x * SV_SMALL_ITEMS;
    const int cnt = (int)((n - base < SV_SMALL_ITEMS) ? (n - base) : SV_SMALL_ITEMS);
    for (int t = threadIdx.x; t < cnt * 32; t += blockDim.x) in_msg[t] = msg[32 * base + t];
    for (int t = threadIdx.x; t < cnt * keylen; t += blockDim.x) in_key[t] = key[(size_t)keylen * base + t];
    for (int t = threadIdx.x; t < cnt * 64; t += blockDim.x) in_sig[t] = sig[64 * base + t];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // phase A (warps 0, 1) and the comb / finish: lane l works on item l; idle lanes redo item 0 into their own slot
    const bool active = lane < cnt;
    const int j = active ? lane : 0;
    sv_small_item* it = &items[lane];
    const u8* m = in_msg + 32 * j;
    const u8* k = in_key + keylen * j;
    const u8* sg = in_sig + 64 * j;
    if constexpr (KIND == SV_KIND_RECOVER) {
        if (warp == 0) small_recover_key_side(sg, k[0], it);   // lift R and tabulate it
        else if (warp == 1) small_recover_scalar_side(m, sg, k[0], it);
    } else {
        if (warp == 0) {
            if (NOSQRT) small_key_side_ns(KIND, k, it); else small_key_side(KIND, k, it);
        } else if (warp == 1) small_scalar_side(KIND, m, k, sg, it);
    }
    __syncthreads();
    // phase B: warps 0..3 run the half ladders on lane PAIRS (warp w: half w >> 1, items 16 (w & 1) + lane / 2), warp 4 the comb
    if (warp < 4) {
        pair_lane L;
        L.role = lane & 1;
        small_half_ladder_pair(L, &items[16 * (warp & 1) + (lane >> 1)], warp >> 1);
    } else {
        small_comb(it, gtab);
    }
    __syncthreads();
    if constexpr (KIND == SV_KIND_RECOVER) {
        if (warp == 0 && active) small_recover_finish(it, k[0], aux + 64 * (base + lane), verdict + base + lane);
    } else if (warp == 0) {
        bool kd = false;
        u32 v = NOSQRT ? small_finish_ns(KIND, it, k, sg, gtab, aux ? &kd : nullptr) : small_finish(KIND, it, sg, &kd);
        if (active) {
            verdict[base + lane] = (u8)v;
            if (aux) aux[base + lane] = (u8)((kd ? 1u : 0u) | ((it->w.flags & SV_WF_PARSED) ? 2u : 0u));
        }
    }
}

// ---- mixed batches (config C3: interleaved ECDSA + BIP-340 with a 1-byte kind tag per item) ---------------------
// The curve kernels are specialised per kind (a warp must be homogeneous), so a mixed batch is split on the DEVICE:
// k_mixed_index appends every item to its kind's index list (warp-aggregated atomics), k_mixed_gather copies each kind's
// items into that kind's dense SoA region, the per-kind kernels run, k_mixed_scatter puts the verdicts back in item order.
__global__ void __launch_bounds__(256) k_mixed_index(const u8* __restrict__ kinds, size_t n, u32* __restrict__ count,
                                                     u32* __restrict__ idx) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    u32 k = (i < n) ? kinds[i] : 3u;
    if (k > 2u) k = 3u;  // unknown kind: no list (verdict stays 0)
    unsigned peers = __match_any_sync(0xFFFFFFFFu, k);
    if (k < 3u) {
        int leader = __ffs(peers) - 1;
        u32 base = 0;
        if ((int)(threadIdx.x & 31) == leader) base = atomicAdd(&count[k], (u32)__popc(peers));
        base = __shfl_sync(peers, base, leader);
        u32 rank = (u32)__popc(peers & ((1u << (threadIdx.x & 31)) - 1u));
        idx[(size_t)k * n + base + rank] = (u32)i;
    }
}
__global__ void __launch_bounds__(256) k_mixed_gather(const u32* __restrict__ idx, size_t c, int keylen,
                                                      const u8* __restrict__ msg, const u8* __restrict__ key64,
                                                      const u8* __restrict__ sig, u8* __restrict__ o_msg,
                                                      u8* __restrict__ o_key, u8* __restrict__ o_sig) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= c) return;
    size_t i = idx[j];
    const uint4* m = reinterpret_cast<const uint4*>(msg + 32 * i);
    const uint4* sg = reinterpret_cast<const uint4*>(sig + 64 * i);
    uint4* om = reinterpret_cast<uint4*>(o_msg + 32 * j);
    uint4* os = reinterpret_cast<uint4*>(o_sig + 64 * j);
    om[0] = m[0]; om[1] = m[1];
    os[0] = sg[0]; os[1] = sg[1]; os[2] = sg[2]; os[3] = sg[3];
    for (int b = 0; b < keylen; b++) o_key[(size_t)keylen * j + b] = key64[64 * i + b];
}
__global__ void __launch_bounds__(256) k_mixed_scatter(const u32* __restrict__ idx, size_t c, const u8* __restrict__ v,
                                                       u8* __restrict__ out) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < c) out[idx[j]] = v[j];
}

// ---- BIP-340 batch verification: the kernels live in batch.cu (compiled with fe_mul / fe_sqr as real functions) ----------
extern "C" int sv_batch_launch(const u8* d_msg, const u8* d_key, const u8* d_sig, size_t n, const u8* d_seed, void* d_pts,
                               signed char* d_dig, void* d_t, u8* d_ok, void* d_S, u8* d_gok, u8* d_out, const void* d_gtab,
                               cudaStream_t st, cudaEvent_t ev_mid);
__global__ void __launch_bounds__(256) k_sb_gather(const u32* __restrict__ idx, size_t c, const u8* __restrict__ msg, const u8* __restrict__ key32,
                                                   const u8* __restrict__ sig, u8* __restrict__ o_msg, u8* __restrict__ o_key, u8* __restrict__ o_sig) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= c) return;
    size_t i = idx[j];
    const uint4* m = reinterpret_cast<const uint4*>(msg + 32 * i);
    const uint4* k = reinterpret_cast<const uint4*>(key32 + 32 * i);
    const uint4* sg = reinterpret_cast<const uint4*>(sig + 64 * i);
    uint4* om = reinterpret_cast<uint4*>(o_msg + 32 * j);
    uint4* ok = reinterpret_cast<uint4*>(o_key + 32 * j);
    uint4* os = reinterpret_cast<uint4*>(o_sig + 64 * j);
    om[0] = m[0]; om[1] = m[1];
    ok[0] = k[0]; ok[1] = k[1];
    os[0] = sg[0]; os[1] = sg[1]; os[2] = sg[2]; os[3] = sg[3];
}

// ---- one key, many signatures (N3): build the key's table once, then a ladder-only curve kernel --------------
__global__ void k_sharedkey_build(int kind, const u8* key, sv_shared_key* out) {
    sharedkey_build(out, kind, key, blockDim.x);  // all 32 lanes compute the same values and store to the same addresses
}
__global__ void __launch_bounds__(SV_MAIN_BLOCK, SV_MAIN_MINB)
    k_main_shared(const sv_work* work, const u8* __restrict__ sig, size_t n, const ge_mem* __restrict__ gtab,
                  const sv_shared_key* sk, const u32* __restrict__ sk_index, u8* __restrict__ verdict, u8* __restrict__ aux) {
    // sk_index == nullptr: ONE key for the whole batch (channeld's HTLC loop); else item i uses table sk[sk_index[i]]
    // (key de-duplication inside a gossip batch: every distinct key is decoded and tabulated once)
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t base = (size_t)blockIdx.x * blockDim.x; base < n; base += stride) {
        size_t i = base + threadIdx.x;
        bool active = i < n;
        const sv_work* w = active ? (work + i) : &g_idle_work;
        const sv_shared_key* k = sk_index ? (sk + sk_index[active ? i : 0]) : sk;
        u32 v = verify_curve_side_shared(w, sig + 64 * (active ? i : 0), gtab, k, blockDim.x);
        if (active) {
            verdict[i] = (u8)v;
            if (aux) aux[i] = (u8)((k->ok ? 1u : 0u) | ((w->flags & SV_WF_PARSED) ? 2u : 0u));
        }
    }
}

// ---- key de-duplication (N3): exact (full 33-byte compare) open-addressing hash table keyed by the key bytes ----
__global__ void __launch_bounds__(256) k_dedup_insert(const u8* __restrict__ key, int keylen, size_t n, u32* slots, u32 mask,
                                                      u32* __restrict__ rep) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u8* k = key + (size_t)keylen * i;
    u32 h = 2166136261u;
    for (int b = 0; b < 12; b++) h = (h ^ k[b]) * 16777619u;  // FNV-1a over the prefix and the top of x
    u32 slot = (h ^ (h >> 15)) & mask;
    for (;;) {
        u32 old = atomicCAS(&slots[slot], 0xFFFFFFFFu, (u32)i);
        if (old == 0xFFFFFFFFu) { rep[i] = (u32)i; return; }
        const u8* o = key + (size_t)keylen * old;
        bool same = true;
        for (int b = 0; b < keylen; b++) same = same && (o[b] == k[b]);
        if (same) { rep[i] = old; return; }
        slot = (slot + 1) & mask;
    }
}
__global__ void __launch_bounds__(256) k_dedup_number(const u32* __restrict__ rep, size_t n, u32* counter, u32* __restrict__ tid,
                                                      u32* __restrict__ replist) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || rep[i] != (u32)i) return;
    u32 t = atomicAdd(counter, 1u);
    tid[i] = t;
    replist[t] = (u32)i;
}
__global__ void __launch_bounds__(256) k_dedup_resolve(const u32* __restrict__ rep, size_t n, u32* __restrict__ tid) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && rep[i] != (u32)i) tid[i] = tid[rep[i]];
}
__global__ void __launch_bounds__(128) k_sharedkey_build_many(int kind, const u8* __restrict__ key, int keylen,
                                                              const u32* __restrict__ replist, u32 distinct, sv_shared_key* out) {
    u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < distinct) sharedkey_build(out + t, kind, key + (size_t)keylen * replist[t]);
}

// ---- device-side BIP143 (SURVEY.md §8f N2): one thread per transaction input -> msg32 ----------------------
__global__ void __launch_bounds__(128) k_bip143(const sv_tx_item* txs, const u8* blob, size_t n, u8* msg32, u8* okout) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    okout[i] = bip143_sighash(msg32 + 32 * i, txs[i], blob) ? 1 : 0;
}
// force verdict 0 where the sighash could not be formed
__global__ void k_mask_verdicts(u8* verdict, const u8* ok, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && !ok[i]) verdict[i] = 0;
}

// ---- gossip ingest (SURVEY.md §8f N1): the device slices raw wire messages itself ----------------------------
// One thread per message.  Field offsets: wire/peer_wire.csv:340-377; signed regions and checking order:
// gossipd/sigcheck.c:9-43 (channel_update), 45-115 (channel_announcement), 118-164 (node_announcement).
// item_base[m] is the first item slot of message m (4 slots for a channel_announcement, 1 otherwise, host-computed
// from the 2-byte type).  Writes span (off,len), key33, sig64 per item; status[m] = -1 if malformed.
__global__ void __launch_bounds__(128) k_gossip_slice(const u8* blob, const u64* msg_off, const u32* msg_len,
                                                      const u32* item_base, const u8* signers33, size_t n_msgs,
                                                      u64* span_off, u32* span_len, u8* key33, u8* sig64, int* status) {
    size_t m = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_msgs) return;
    const u8* p = blob + msg_off[m];
    u32 len = msg_len[m];
    u32 type = len >= 2 ? (((u32)p[0] << 8) | p[1]) : 0;
    u32 base = item_base[m];
    int nitems = (type == 256) ? 4 : ((type == 257 || type == 258) ? 1 : 0);
    int st = 0;
    u32 hoff = (type == 256) ? 258 : 66;
    u32 keys = 0;
    if (type == 256) {
        if (len < 260) st = -1;
        else {
            u32 flen = ((u32)p[258] << 8) | p[259];
            keys = 260 + flen + 32 + 8;
            if (len < keys + 4 * 33) st = -1;
        }
    } else if (type == 257) {
        // signature(64) flen(2) features timestamp(4) node_id(33) rgb_color(3) alias(32) addrlen(2) addresses
        // (wire/peer_wire.csv:353-362): fromwire_node_announcement fails on any shorter message
        if (len < 68) st = -1;
        else {
            u32 flen = ((u32)p[66] << 8) | p[67];
            keys = 68 + flen + 4;
            if (len < keys + 33 + 3 + 32 + 2) st = -1;
            else {
                u32 alen = ((u32)p[keys + 68] << 8) | p[keys + 69];
                if (len < keys + 70 + alen) st = -1;
            }
        }
    } else if (type == 258) {
        // signature(64) chain_hash(32) short_channel_id(8) timestamp(4) message_flags(1) channel_flags(1)
        // cltv_expiry_delta(2) htlc_minimum_msat(8) fee_base_msat(4) fee_proportional_millionths(4)
        // htlc_maximum_msat(8) = 138 bytes with the type (wire/peer_wire.csv:366-377; htlc_maximum_msat is mandatory)
        if (len < 138 || signers33 == nullptr) st = -1;
    } else {
        st = -1;
    }
    for (int k = 0; k < nitems; k++) {
        u32 it = base + k;
        bool ok = (st == 0);
        span_off[it] = msg_off[m] + (ok ? hoff : 0);
        span_len[it] = ok ? (len - hoff) : 0;
        const u8* kp = (type == 258) ? (signers33 ? signers33 + 33 * m : p) : (p + keys + 33 * k);
        for (int b = 0; b < 33; b++) key33[33 * (size_t)it + b] = ok ? kp[b] : 0;  // an all-zero key never verifies
        const u8* sp = p + 2 + 64 * k;
        for (int b = 0; b < 64; b++) sig64[64 * (size_t)it + b] = ok ? sp[b] : 0;
    }
    status[m] = st;
}
// status[m] = 1 + index of the first failing signature (the reference's order), 0 if all verify
// -1 also when CLN's wire parser would refuse the message: a signature with r >= n or s >= n
// (fromwire_secp256k1_ecdsa_signature, wire/fromwire.c:188-199) or an undecodable bitcoin_key (fromwire_pubkey,
// bitcoin/pubkey.c:102-113).  node_ids are raw bytes on the wire (common/node_id.c:54) and only fail the signature.
__global__ void __launch_bounds__(128) k_gossip_status(const u8* blob, const u64* msg_off, const u32* msg_len,
                                                       const u32* item_base, size_t n_msgs, const u8* verdict,
                                                       const u8* aux, int* status) {
    size_t m = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_msgs || status[m] != 0) return;
    const u8* p = blob + msg_off[m];
    u32 type = ((u32)p[0] << 8) | p[1];
    int nitems = (type == 256) ? 4 : 1;
    int st = 0;
    for (int k = nitems - 1; k >= 0; k--)
        if (!verdict[item_base[m] + k]) st = k + 1;
    for (int k = 0; k < nitems; k++) {
        u32 it = item_base[m] + k;
        if (!(aux[it] & 2u)) st = -1;                           // r or s >= n: the wire parser refuses the message
        if (type == 256 && k >= 2 && !(aux[it] & 1u)) st = -1;  // undecodable bitcoin_key
    }
    status[m] = st;
}

static_assert(sizeof(sv_jac) == sizeof(sv_work), "R is parked in place of the work record");
__global__ void __launch_bounds__(64) k_final_schnorr(const sv_work* work, const u8* sig, size_t n, u8* verdict) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t base = t * SV_FINAL_BATCH;
    if (base >= n) return;
    int cnt = (int)((n - base < SV_FINAL_BATCH) ? (n - base) : SV_FINAL_BATCH);
    schnorr_final_batch(verdict + base, reinterpret_cast<const sv_jac*>(work) + base, sig + 64 * base, cnt);
}

// public-key recovery: affine keys from the parked Q (batched inversion), status 1 / 0 / -1 as a byte
__global__ void __launch_bounds__(64) k_final_recover(const sv_work* work, size_t n, u8* xy64, u8* status) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t base = t * SV_FINAL_BATCH;
    if (base >= n) return;
    int cnt = (int)((n - base < SV_FINAL_BATCH) ? (n - base) : SV_FINAL_BATCH);
    recover_final_batch(xy64 + 64 * base, status + base, reinterpret_cast<const sv_jac*>(work) + base, cnt);
}

static_assert(sizeof(sv_ns_park) == sizeof(sv_work), "D, B, c are parked in place of the work record");
__global__ void __launch_bounds__(64) k_final_ecdsa33(const sv_work* work, const u8* key33, const u8* sig, size_t n,
                                                       const ge_mem* gtab, u8* verdict, u8* aux) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t base = t * SV_FINAL_BATCH;
    if (base >= n) return;
    int cnt = (int)((n - base < SV_FINAL_BATCH) ? (n - base) : SV_FINAL_BATCH);
    ecdsa33_nosqrt_final_batch(verdict + base, work + base, key33 + 33 * base, sig + 64 * base, gtab, cnt, aux ? aux + base : nullptr);
}

static_assert(sizeof(sv_ns_park_schnorr) == sizeof(sv_work), "D, B, N, CG are parked in place of the work record");
__global__ void __launch_bounds__(64) k_final_schnorr_ns(const sv_work* work, const u8* xonly32, const u8* sig, size_t n,
                                                          const ge_mem* gtab, u8* verdict) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t base = t * SV_FINAL_BATCH;
    if (base >= n) return;
    int cnt = (int)((n - base < SV_FINAL_BATCH) ? (n - base) : SV_FINAL_BATCH);
    schnorr_nosqrt_final_batch(verdict + base, work + base, xonly32 + 32 * base, sig + 64 * base, gtab, cnt);
}

__global__ void k_pack_bitmap(const u8* verdict, size_t n, u32* bitmap) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    u32 v = (i < n) ? (verdict[i] != 0) : 0u;
    u32 b = __ballot_sync(0xFFFFFFFFu, v);
    if ((threadIdx.x & 31) == 0 && i < n) bitmap[i >> 5] = b;
}

__global__ void __launch_bounds__(128) k_pubkey_parse(const u8* key33, size_t n, u8* xy64, u8* okout) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ge Q;
    bool ok = key_decode(Q, SV_KIND_ECDSA33, key33 + 33 * i);
    if (ok) {
        fe_get_b32(xy64 + 64 * i, Q.x);
        fe_get_b32(xy64 + 64 * i + 32, Q.y);
    } else {
        for (int k = 0; k < 64; k++) xy64[64 * i + k] = 0;
    }
    okout[i] = ok;
}

// ---- device-side self test of the arithmetic primitives (test support; body in selftest.cuh) -------
__global__ void __launch_bounds__(128) k_selftest(int op, const u32* __restrict__ a, const u32* __restrict__ b, size_t n,
                                                  u32* __restrict__ out, const ge_mem* __restrict__ gtab) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 A[8], B[8], R[16];
#pragma unroll
    for (int k = 0; k < 8; k++) { A[k] = a[8 * i + k]; B[k] = b[8 * i + k]; }
    selftest_item(op, A, B, R, gtab);
#pragma unroll
    for (int k = 0; k < 16; k++) out[16 * i + k] = R[k];
}

// ---- synthetic workload generator ---------------------------------------------------------------
SV_D void synth_hash(u8 out[32], u64 seed, u64 idx, u32 tag) {
    u8 buf[20];
    for (int k = 0; k < 8; k++) { buf[k] = (u8)(seed >> (8 * k)); buf[8 + k] = (u8)(idx >> (8 * k)); }
    for (int k = 0; k < 4; k++) buf[16 + k] = (u8)(tag >> (8 * k));
    u32 st[8];
    sha256_bytes(st, buf, 20);
    for (int k = 0; k < 8; k++) {
        out[4 * k] = (u8)(st[k] >> 24); out[4 * k + 1] = (u8)(st[k] >> 16);
        out[4 * k + 2] = (u8)(st[k] >> 8); out[4 * k + 3] = (u8)st[k];
    }
}
template <int KIND>
__global__ void __launch_bounds__(128) k_synth(u64 seed, size_t n, const ge_mem* gtab, u8* msg, u8* key, u8* sig) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u8 h[32];
    sc d, k, m, one;
#pragma unroll
    for (int q = 0; q < 8; q++) one.v[q] = (q == 0);
    synth_hash(h, seed, i, 1);
    sc_set_b32(d, h, nullptr);
    if (sc_is_zero(d)) d = one;
    synth_hash(h, seed, i, 2);
    sc_set_b32(k, h, nullptr);
    if (sc_is_zero(k)) k = one;
    synth_hash(h, seed, i, 3);
    for (int q = 0; q < 32; q++) msg[32 * i + q] = h[q];
    sc_set_b32(m, h, nullptr);
    ge P, R;
    ecmult_gen_comb(P, d, gtab);
    ecmult_gen_comb(R, k, gtab);
    if (KIND == SV_KIND_SCHNORR) {
        // BIP-340 signing equation with even-y P and R: s = k + e*d
        if (fe_is_odd(P.y)) sc_negate(d, d);
        if (fe_is_odd(R.y)) sc_negate(k, k);
        u8 rx[32], px[32], e32[32];
        fe_get_b32(rx, R.x);
        fe_get_b32(px, P.x);
        sha256_bip340_challenge(e32, rx, px, h);
        sc e, s;
        sc_set_b32(e, e32, nullptr);
        sc_mul(s, e, d);
        sc_add(s, s, k);
        for (int q = 0; q < 32; q++) { key[32 * i + q] = px[q]; sig[64 * i + q] = rx[q]; }
        sc_get_b32(sig + 64 * i + 32, s);
    } else {
        // ECDSA: r = x(kG) mod n, s = (m + r d)/k, normalised to low S
        u8 rx[32];
        fe_get_b32(rx, R.x);
        sc r, s, kinv;
        sc_set_b32(r, rx, nullptr);
        sc_inverse(kinv, k);
        sc_mul(s, r, d);
        sc_add(s, s, m);
        sc_mul(s, s, kinv);
        if (sc_is_high(s)) sc_negate(s, s);
        sc_get_b32(sig + 64 * i, r);
        sc_get_b32(sig + 64 * i + 32, s);
        if (KIND == SV_KIND_ECDSA33) {
            key[33 * i] = fe_is_odd(P.y) ? 3 : 2;
            fe_get_b32(key + 33 * i + 1, P.x);
        } else {
            fe_get_b32(key + 64 * i, P.x);
            fe_get_b32(key + 64 * i + 32, P.y);
        }
    }
}

// ---- integer-pipe probes ------------------------------------------------------------------------
// Each probe is its own kernel so that ncu reports them separately.  All run 256 threads x 8 CTAs/SM.
//   0 k_probe_imad_wide   independent IMAD.WIDE.U32 accumulations (no carries)      -> MAC/s (roofline peak)
//   1 k_probe_cmad4       4-deep IMAD.WIDE.U32(.X) carry chains as u256_mul_wide issues them -> MAC/s
//   2 k_probe_fe_mul      field multiplications/s          3 k_probe_fe_sqr   field squarings/s
//   4 k_probe_chain8      8-deep IMAD.WIDE.U32.X chains    -> MAC/s
//   5 k_probe_carry_save  IMAD.WIDE.U32 with carry-OUT only + one IADD3.X per product -> MAC/s
//   6 k_probe_imad32      separate 32-bit IMAD (lo) / IMAD.HI  -> instr/s
//   7 k_probe_addc        8-long IADD3(.X) carry chains -> adds/s
//   8 k_probe_dfma        independent FP64 FMA chains -> DFMA/s (the idle FP64 pipe; round-2 idea: DFMA-based products)
#define PROBE_PROLOGUE u32 t = blockIdx.x * blockDim.x + threadIdx.x
__global__ void __launch_bounds__(256) k_probe_imad_wide(int iters, u32* sink) {
    PROBE_PROLOGUE;
    u32 lo[8], hi[8];
#pragma unroll
    for (int k = 0; k < 8; k++) { lo[k] = t * 2654435761u + k; hi[k] = t ^ (k * 0x9E3779B9u); }
    u32 y = t | 3u;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int r = 0; r < 4; r++) {
            // acc_k += lo(acc_{k+1}) * y : eight independent 64-bit multiply-accumulates per step whose
            // multiplicands change every step (so ptxas cannot strength-reduce them to additions)
#pragma unroll
            for (int k = 0; k < 8; k++)
                asm volatile("mad.lo.cc.u32 %0, %2, %3, %0;\n\tmadc.hi.u32 %1, %2, %3, %1;"
                             : "+r"(lo[k]), "+r"(hi[k])
                             : "r"(lo[(k + 1) & 7]), "r"(y));
        }
    }
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= lo[k] ^ hi[k];
    if (s == 0x1234567u) sink[0] = s;
}
__global__ void __launch_bounds__(256) k_probe_cmad4(int iters, u32* sink) {
    PROBE_PROLOGUE;
    u32 E[8], O[8];
#pragma unroll
    for (int k = 0; k < 8; k++) { E[k] = t + k; O[k] = t * 3 + k; }
    u32 a0 = t | 1, a1 = t ^ 0xABCDEFu, a2 = t * 7 + 1, a3 = ~t, b = t * 2654435761u;
    u32 cs = 0;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
            cs += sv_cmad4(E, a0, a1, a2, a3, b);
            cs += sv_cmad4(O, a1, a2, a3, a0, b);
        }
    }
    u32 s = cs;
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= E[k] ^ O[k];
    if (s == 0x12345u) sink[0] = s;
}
template <int SQR>
__global__ void __launch_bounds__(256) k_probe_fe(int iters, u32* sink) {
    PROBE_PROLOGUE;
    fe a, b;
#pragma unroll
    for (int k = 0; k < 8; k++) { a.v[k] = t * 2654435761u + k; b.v[k] = (t ^ 0x5bd1e995u) * (k + 3); }
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
        if (!SQR) { fe_mul(a, a, b); fe_mul(b, b, a); }
        else { fe_sqr(a, a); fe_sqr(b, b); }
    }
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= a.v[k] ^ b.v[k];
    if (s == 0x12345u) sink[0] = s;
}
__global__ void __launch_bounds__(256) k_probe_chain8(int iters, u32* sink) {
    PROBE_PROLOGUE;
    u32 A[16], B[16];
#pragma unroll
    for (int k = 0; k < 16; k++) { A[k] = t + k; B[k] = t * 5 + k; }
    u32 x0 = t | 1, x1 = t ^ 0xABCDEFu, x2 = t * 7 + 1, x3 = ~t, y = t * 2654435761u;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 2; k++) {
#define CHAIN8(ACC)                                                                                              \
    asm volatile("mad.lo.cc.u32 %0, %16, %20, %0;\n\tmadc.hi.cc.u32 %1, %16, %20, %1;\n\t"                         \
                 "madc.lo.cc.u32 %2, %17, %20, %2;\n\tmadc.hi.cc.u32 %3, %17, %20, %3;\n\t"                        \
                 "madc.lo.cc.u32 %4, %18, %20, %4;\n\tmadc.hi.cc.u32 %5, %18, %20, %5;\n\t"                        \
                 "madc.lo.cc.u32 %6, %19, %20, %6;\n\tmadc.hi.cc.u32 %7, %19, %20, %7;\n\t"                        \
                 "madc.lo.cc.u32 %8, %17, %20, %8;\n\tmadc.hi.cc.u32 %9, %17, %20, %9;\n\t"                        \
                 "madc.lo.cc.u32 %10, %18, %20, %10;\n\tmadc.hi.cc.u32 %11, %18, %20, %11;\n\t"                    \
                 "madc.lo.cc.u32 %12, %19, %20, %12;\n\tmadc.hi.cc.u32 %13, %19, %20, %13;\n\t"                    \
                 "madc.lo.cc.u32 %14, %16, %20, %14;\n\tmadc.hi.u32 %15, %16, %20, %15;"                           \
                 : "+r"(ACC[0]), "+r"(ACC[1]), "+r"(ACC[2]), "+r"(ACC[3]), "+r"(ACC[4]), "+r"(ACC[5]), "+r"(ACC[6]), \
                   "+r"(ACC[7]), "+r"(ACC[8]), "+r"(ACC[9]), "+r"(ACC[10]), "+r"(ACC[11]), "+r"(ACC[12]),           \
                   "+r"(ACC[13]), "+r"(ACC[14]), "+r"(ACC[15])                                                      \
                 : "r"(x0), "r"(x1), "r"(x2), "r"(x3), "r"(y))
            CHAIN8(A);
            CHAIN8(B);
        }
    }
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) s ^= A[k] ^ B[k];
    if (s == 0x12345u) sink[0] = s;
}
__global__ void __launch_bounds__(256) k_probe_carry_save(int iters, u32* sink) {
    PROBE_PROLOGUE;
    u32 lo[8], hi[8], c[8];
#pragma unroll
    for (int k = 0; k < 8; k++) { lo[k] = t + k; hi[k] = t * 3 + k; c[k] = k; }
    u32 x = t * 2654435761u + 12345u, y = t ^ 0x9E3779B9u;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int r = 0; r < 4; r++) {
#pragma unroll
            for (int k = 0; k < 8; k++)
                asm volatile("mad.lo.cc.u32 %0, %3, %4, %0;\n\tmadc.hi.cc.u32 %1, %3, %4, %1;\n\taddc.u32 %2, %2, 0;"
                             : "+r"(lo[k]), "+r"(hi[k]), "+r"(c[k])
                             : "r"(x), "r"(y));
        }
    }
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= lo[k] ^ hi[k] ^ c[k];
    if (s == 0x12345u) sink[0] = s;
}
__global__ void __launch_bounds__(256) k_probe_imad32(int iters, u32* sink) {
    PROBE_PROLOGUE;
    u32 a[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = t + k;
    u32 x = t * 2654435761u + 12345u, y = t ^ 0x9E3779B9u, z = t * 31 + 7;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int r = 0; r < 4; r++) {
#pragma unroll
            for (int k = 0; k < 8; k += 2)
                asm volatile("mad.lo.u32 %0, %2, %3, %0;\n\tmad.hi.u32 %1, %2, %4, %1;"
                             : "+r"(a[k]), "+r"(a[k + 1])
                             : "r"(x), "r"(y), "r"(z));
        }
    }
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= a[k];
    if (s == 0x12345u) sink[0] = s;
}
__global__ void __launch_bounds__(256) k_probe_dfma(int iters, u32* sink) {
    PROBE_PROLOGUE;
    double a[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = 1.0 + (double)(t + k) * 1e-9;
    double x = 1.0000001 + (double)t * 1e-12, y = 0.9999999;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int r = 0; r < 4; r++) {
#pragma unroll
            for (int k = 0; k < 8; k++) a[k] = fma(a[k], x, y);
        }
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += a[k];
    if (s == 1234.5) sink[0] = 1;
}
__global__ void __launch_bounds__(256) k_probe_addc(int iters, u32* sink) {
    PROBE_PROLOGUE;
    u32 a[8], b[8], c[8], d[8];
#pragma unroll
    for (int k = 0; k < 8; k++) { a[k] = t + k; b[k] = t * 3 + k; c[k] = t ^ k; d[k] = ~t + k; }
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int r = 0; r < 2; r++) {
            u256_add(a, a, b);
            u256_add(c, c, d);
            u256_add(b, b, c);
            u256_add(d, d, a);
        }
    }
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= a[k] ^ b[k] ^ c[k] ^ d[k];
    if (s == 0x12345u) sink[0] = s;
}

// -------------------------------------------------------------------------------------------------
// context
// -------------------------------------------------------------------------------------------------
#define SV_NSLOTS 2
#define SV_SMALL_CAP 8192           // items the pinned small-batch staging block holds
#ifndef SV_SMALL_MAX_DEFAULT
// largest batch sent down the small-batch path (SV_SMALL_MAX overrides; 0 disables).  Measured (profiles/r2_latency_paths_1k_8k.txt):
// 4,096 signatures 480 us against 1,248 us on the throughput kernels, 8,192 signatures 661 against 1,272 us
#define SV_SMALL_MAX_DEFAULT 8192
#endif
struct sv_queue_item {
    int kind;
    u8 msg[32];
    u8 key[64];
    u8 sig[64];
};

struct sv_ctx {
    int device;
    int sm_count;
    cudaStream_t stream;
    cudaStream_t stream2;      // second compute stream: consecutive slices of a large host batch alternate streams, so the
                               // thin last wave of one slice's curve kernel overlaps the next slice's kernels
    cudaStream_t copy_stream;  // H2D of the next slice overlaps the kernels of the current one (sv_verify_host)
    cudaEvent_t h2d_ev[8];
    ge_mem* d_gtab;
    u8* d_hot;          // [G comb table | slot 0 table slab | slot 1 table slab]
    size_t hot_bytes, l2_persist, l2_max_persist, hot_slab, hot_gt;
    cudaStream_t policy_streams[4];  // (stream, slab) pairs whose access-policy window is already set
    const void* policy_slabs[4];
    int l2_policy;      // sv_set_l2_policy (default on)
    ge_mem* d_bases;
    size_t scratch_bytes;
    int main_grid;
    // Launch slots: the scalar-side work records and the per-thread Q-table slab of one prep+main launch pair.  Two slots,
    // used round-robin, let launches issued on DIFFERENT streams overlap (the partially filled last wave of one batch's
    // curve kernel runs beside the next batch's kernels); a slot is re-used only after the event recorded behind its
    // previous use, so calls on one context can never corrupt each other whatever streams the caller picks.
    struct slot_t {
        sv_work* d_work;
        size_t work_cap;
        qtab_entry* d_scratch;
        cudaEvent_t done;
        cudaStream_t last_stream;
        int used;
    } slot[SV_NSLOTS];
    unsigned next_slot;
    // small-batch path: calls of up to small_max signatures run as ONE launch of k_small reading their inputs straight
    // from this pinned, device-mapped staging block (no H2D/D2H copy commands, no allocation)
    size_t small_max, small_cap;
    u8* h_small;
    // key de-duplication scratch (hash table + index lists) and the table array of the distinct keys, grow-only
    u8 *dd_buf, *sk_buf;
    size_t dd_cap, sk_cap;
    int dedup;  // gossip batches: look for repeated keys (sv_set_dedup; default on)
    int nosqrt; // compressed-key ECDSA through the flow without the square root (default on; env SV_NOSQRT=0: measurement aid)
    u32 last_distinct;
    // growable device staging for the host-buffer entry points
    size_t cap;  // items
    u8 *d_msg, *d_key, *d_sig, *d_verdict;
    // raw-span staging
    u8* d_data;
    size_t data_cap;
    u64* d_off;
    u32* d_len;
    size_t span_cap;
    u32* d_sink;
    // gossip ingest scratch (grow-only)
    u8* g_buf;
    size_t g_cap;
    int profiling;
    cudaEvent_t ev[3];  // before prep, between prep and main, after main (profiling mode only)
    unsigned long long launches;
    std::vector<sv_queue_item> queue;
    std::string err;
};

static std::string g_create_err;

// temporary device allocation released on every exit path
struct dev_tmp {
    void* p = nullptr;
    ~dev_tmp() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};

// every entry point runs on the context's device and puts the caller's current device back on return
struct dev_guard {
    int prev = -1;
    cudaError_t enter(int dev) {
        cudaError_t e = cudaGetDevice(&prev);
        if (e != cudaSuccess) { prev = -1; return e; }
        if (prev == dev) { prev = -1; return cudaSuccess; }
        return cudaSetDevice(dev);
    }
    ~dev_guard() { if (prev >= 0) cudaSetDevice(prev); }
};

static int fail(sv_ctx* ctx, int code, const char* what, cudaError_t e) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s", what, e == cudaSuccess ? "" : cudaGetErrorString(e));
    if (ctx) ctx->err = buf; else g_create_err = buf;
    return code;
}
#define CK(call)                                                                   \
    do {                                                                           \
        cudaError_t e__ = (call);                                                  \
        if (e__ != cudaSuccess) return fail(ctx, e__ == cudaErrorMemoryAllocation ? SV_ERR_NOMEM : SV_ERR_CUDA, #call, e__); \
    } while (0)

extern "C" size_t sv_key_size(int kind) {
    return kind == SV_KIND_ECDSA33 ? 33 : kind == SV_KIND_ECDSA_XY ? 64 : kind == SV_KIND_SCHNORR ? 32 : 0;
}
extern "C" const char* sv_last_error(const sv_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

// Pick the next launch slot for n work records on stream st: waits (on the device, not the host) for the slot's previous
// user if that ran on another stream, grows the record array geometrically when needed (the only host-synchronising case).
static int acquire_slot(sv_ctx* ctx, size_t n, cudaStream_t st, sv_ctx::slot_t** out) {
    sv_ctx::slot_t* sl = &ctx->slot[ctx->next_slot++ % SV_NSLOTS];
    if (sl->used && sl->last_stream != st) CK(cudaStreamWaitEvent(st, sl->done, 0));
    if (n > sl->work_cap) {
        if (sl->used) CK(cudaEventSynchronize(sl->done));
        size_t cap = sl->work_cap ? sl->work_cap : 4096;
        while (cap < n) cap *= 2;
        if (sl->d_work) cudaFree(sl->d_work);
        sl->d_work = nullptr;
        sl->work_cap = 0;
        CK(cudaMalloc(&sl->d_work, cap * sizeof(sv_work)));
        sl->work_cap = cap;
    }
    *out = sl;
    return SV_OK;
}
static int release_slot(sv_ctx* ctx, sv_ctx::slot_t* sl, cudaStream_t st) {
    CK(cudaEventRecord(sl->done, st));
    sl->last_stream = st;
    sl->used = 1;
    return SV_OK;
}
static int ensure_staging(sv_ctx* ctx, size_t n) {
    if (n <= ctx->cap) return SV_OK;
    CK(cudaDeviceSynchronize());  // growth only: in-flight launches may still read the old buffers
    size_t want = ctx->cap ? ctx->cap : 4096;
    while (want < n) want *= 2;
    n = want;
    cudaFree(ctx->d_msg); cudaFree(ctx->d_key); cudaFree(ctx->d_sig); cudaFree(ctx->d_verdict);
    ctx->d_msg = ctx->d_key = ctx->d_sig = ctx->d_verdict = nullptr;
    ctx->cap = 0;
    CK(cudaMalloc(&ctx->d_msg, n * 32));
    CK(cudaMalloc(&ctx->d_key, n * 64));
    CK(cudaMalloc(&ctx->d_sig, n * 64));
    CK(cudaMalloc(&ctx->d_verdict, n));
    ctx->cap = n;
    return SV_OK;
}

extern "C" int sv_create(sv_ctx** out, int device) {
    sv_ctx* ctx = nullptr;
    if (!out) return SV_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return fail(nullptr, SV_ERR_NO_DEVICE, "no CUDA device (this engine has no CPU fallback)", e);
    if (device < 0 || device >= ndev) return fail(nullptr, SV_ERR_ARG, "bad device ordinal", cudaSuccess);
    dev_guard dg__;
    CK(dg__.enter(device));
    ctx = new sv_ctx();
    ctx->device = device;
    ctx->cap = ctx->data_cap = ctx->span_cap = 0;
    for (int i = 0; i < SV_NSLOTS; i++) { ctx->slot[i].d_work = nullptr; ctx->slot[i].work_cap = 0; ctx->slot[i].d_scratch = nullptr;
                                          ctx->slot[i].done = nullptr; ctx->slot[i].last_stream = nullptr; ctx->slot[i].used = 0; }
    ctx->next_slot = 0;
    ctx->d_hot = nullptr;
    ctx->hot_bytes = ctx->l2_persist = ctx->l2_max_persist = ctx->hot_slab = ctx->hot_gt = 0;
    ctx->l2_policy = 1;
    if (const char* e = getenv("SV_L2_POLICY")) ctx->l2_policy = atoi(e) != 0;  // measurement aid
    for (int i = 0; i < 4; i++) { ctx->policy_streams[i] = nullptr; ctx->policy_slabs[i] = nullptr; }
    ctx->h_small = nullptr;
    ctx->dd_buf = ctx->sk_buf = nullptr;
    ctx->dd_cap = ctx->sk_cap = 0;
    ctx->dedup = 1;
    ctx->nosqrt = 1;
    if (const char* e = getenv("SV_NOSQRT")) ctx->nosqrt = atoi(e) != 0;
    ctx->last_distinct = 0;
    ctx->small_cap = SV_SMALL_CAP;
    ctx->small_max = SV_SMALL_MAX_DEFAULT;
    if (const char* e = getenv("SV_SMALL_MAX")) ctx->small_max = (size_t)strtoull(e, nullptr, 10);
    if (ctx->small_max > ctx->small_cap) ctx->small_max = ctx->small_cap;
    ctx->d_msg = ctx->d_key = ctx->d_sig = ctx->d_verdict = ctx->d_data = nullptr;
    ctx->d_off = nullptr; ctx->d_len = nullptr;
    ctx->launches = 0;
    ctx->g_buf = nullptr;
    ctx->g_cap = 0;
    ctx->profiling = 0;
    ctx->ev[0] = ctx->ev[1] = ctx->ev[2] = nullptr;
    ctx->stream = ctx->stream2 = ctx->copy_stream = nullptr;
    for (int i = 0; i < 8; i++) ctx->h2d_ev[i] = nullptr;
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) { int rc = fail(nullptr, SV_ERR_CUDA, "cudaGetDeviceProperties", e); delete ctx; return rc; }
    ctx->sm_count = prop.multiProcessorCount;
    int rc = SV_OK;
    do {
#define CK2(call) { cudaError_t e2 = (call); if (e2 != cudaSuccess) { rc = fail(nullptr, e2 == cudaErrorMemoryAllocation ? SV_ERR_NOMEM : SV_ERR_CUDA, #call, e2); break; } }
        CK2(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        CK2(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
        CK2(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 8 && rc == SV_OK; i++) CK2(cudaEventCreateWithFlags(&ctx->h2d_ev[i], cudaEventDisableTiming));
        if (rc != SV_OK) break;
        // G table and the launch slots' per-thread table slabs live in ONE allocation: a single L2 access-policy window
        // then covers everything the curve kernel reads more than once (see apply_l2_policy)
        CK2(cudaMalloc(&ctx->d_bases, 16 * sizeof(ge_mem)));
        CK2(cudaMalloc(&ctx->d_sink, 64));
        CK2(cudaHostAlloc((void**)&ctx->h_small, (size_t)SV_SMALL_CAP * (32 + 64 + 64 + 2), cudaHostAllocMapped | cudaHostAllocPortable));
        int occ = 0;
        CK2(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_main<SV_KIND_ECDSA33>, SV_MAIN_BLOCK, SV_MAIN_SMEM));
        if (occ < 1) occ = 1;
        ctx->main_grid = ctx->sm_count * occ;
        // deployment knob: leave a few CTA slots of the persistent curve kernel free for a collective's kernel that becomes
        // ready while the grid is resident (bench.py sets 2 when it gathers verdict bitmaps over NCCL)
        if (const char* e = getenv("SV_MAIN_GRID_RESERVE")) {
            int r = atoi(e);
            if (r > 0 && r < ctx->main_grid) ctx->main_grid -= r;
        }
        ctx->scratch_bytes = (size_t)ctx->main_grid * SV_MAIN_BLOCK * 8 * sizeof(qtab_entry);
        {
            size_t gt = ((size_t)SV_GT_ENTRIES * sizeof(ge_mem) + 255) & ~(size_t)255;
            size_t sb = (ctx->scratch_bytes + 255) & ~(size_t)255;
            ctx->hot_bytes = gt + SV_NSLOTS * sb;
            CK2(cudaMalloc(&ctx->d_hot, ctx->hot_bytes));
            // layout [slab 0 | G table | slab 1]: each slot's slab is contiguous with the G table, so one window covers both
            static_assert(SV_NSLOTS == 2, "the hot-region layout below is for two launch slots");
            ctx->slot[0].d_scratch = reinterpret_cast<qtab_entry*>(ctx->d_hot);
            ctx->d_gtab = reinterpret_cast<ge_mem*>(ctx->d_hot + sb);
            ctx->slot[1].d_scratch = reinterpret_cast<qtab_entry*>(ctx->d_hot + sb + gt);
            ctx->hot_slab = sb;
            ctx->hot_gt = gt;
            // persisting L2 carve-out (as much as the device allows); failure is not an error: the hint is then simply absent
            int maxp = 0;
            if (cudaDeviceGetAttribute(&maxp, cudaDevAttrMaxPersistingL2CacheSize, device) == cudaSuccess && maxp > 0 &&
                cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)maxp < sb + gt ? (size_t)maxp : sb + gt) == cudaSuccess)
                ctx->l2_persist = (size_t)maxp < sb + gt ? (size_t)maxp : sb + gt;  // one slab + the G table; the rest of L2 stays ordinary
            else (void)cudaGetLastError();
            ctx->l2_max_persist = maxp > 0 ? (size_t)maxp : 0;
        }
        for (int i = 0; i < SV_NSLOTS && rc == SV_OK; i++) CK2(cudaEventCreateWithFlags(&ctx->slot[i].done, cudaEventDisableTiming));
        if (rc != SV_OK) break;
        k_gtable_bases<<<1, 32, 0, ctx->stream>>>(ctx->d_bases);
        k_gtable_fill<<<(SV_GT_ENTRIES + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_gtab, ctx->d_bases);
        ctx->launches += 2;
        CK2(cudaGetLastError());
#ifdef SV_COMB_SMEM
        {
            ge_mem* t8 = nullptr;
            CK2(cudaMalloc(&t8, 17 * 128 * sizeof(ge_mem)));
            k_t8_fill<<<17, 128, 0, ctx->stream>>>(t8, ctx->d_gtab);
            CK2(cudaMemcpyToSymbolAsync(g_t8, &t8, sizeof(t8), 0, cudaMemcpyHostToDevice, ctx->stream));
            const int smem = 17 * 128 * (int)sizeof(ge_mem);
            CK2(cudaFuncSetAttribute(k_main<SV_KIND_ECDSA33>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            CK2(cudaFuncSetAttribute(k_main<SV_KIND_ECDSA_XY>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            CK2(cudaFuncSetAttribute(k_main<SV_KIND_SCHNORR>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        }
#endif
        CK2(cudaStreamSynchronize(ctx->stream));
#undef CK2
    } while (0);
    if (rc != SV_OK) { sv_destroy(ctx); return rc; }
    *out = ctx;
    return SV_OK;
}

extern "C" void sv_destroy(sv_ctx* ctx) {
    if (!ctx) return;
    dev_guard dg__;
    dg__.enter(ctx->device);
    cudaDeviceSynchronize();
    cudaFree(ctx->d_hot); cudaFree(ctx->d_bases); cudaFree(ctx->d_sink);
    if (ctx->h_small) cudaFreeHost(ctx->h_small);
    cudaFree(ctx->dd_buf); cudaFree(ctx->sk_buf);
    for (int i = 0; i < SV_NSLOTS; i++) {
        cudaFree(ctx->slot[i].d_work);
        if (ctx->slot[i].done) cudaEventDestroy(ctx->slot[i].done);
    }
    cudaFree(ctx->d_msg); cudaFree(ctx->d_key); cudaFree(ctx->d_sig); cudaFree(ctx->d_verdict);
    cudaFree(ctx->d_data); cudaFree(ctx->d_off); cudaFree(ctx->d_len); cudaFree(ctx->g_buf);
    for (int i = 0; i < 3; i++) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < 8; i++) if (ctx->h2d_ev[i]) cudaEventDestroy(ctx->h2d_ev[i]);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" int sv_get_info(const sv_ctx* ctx, sv_info* info) {
    if (!ctx || !info) return SV_ERR_ARG;
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, k_main<SV_KIND_ECDSA33>);
    info->device = ctx->device;
    info->sm_count = ctx->sm_count;
    info->main_block = SV_MAIN_BLOCK;
    info->main_grid = ctx->main_grid;
    info->main_regs = fa.numRegs;
    info->gtable_bytes = (size_t)SV_GT_ENTRIES * sizeof(ge_mem);
    info->scratch_bytes = ctx->scratch_bytes;
    info->l2_persist_bytes = ctx->l2_policy ? ctx->l2_persist : 0;
    info->l2_max_persist_bytes = ctx->l2_max_persist;
    info->launches = ctx->launches;
    return SV_OK;
}

// launch prep + main on device-resident SoA arrays.  *used (optional) receives the slot whose work records the launch
// wrote (the gossip status kernel reads their flags afterwards, on the same stream).
// ECDSA batch with repeated keys: returns 1 if it handled the batch (enough repetition to pay), 0 if the caller should take
// the ordinary path, < 0 on error.  Synchronises the stream once (the number of distinct keys sizes the table array).
static int launch_verify_dedup(sv_ctx* ctx, int kind, const u8* d_msg, const u8* d_key, const u8* d_sig, size_t n,
                               u8* d_verdict, cudaStream_t st, u8* d_aux, u32* distinct_out) {
    // batches the small-batch kernel takes are faster there than through the search (one launch, ~0.5 ms)
    if (kind == SV_KIND_SCHNORR || n < 4096 || n <= ctx->small_max || n > 0x7FFFFFFFu) return 0;
    const int keylen = (int)sv_key_size(kind);
    u32 cap = 1;
    while (cap < 2 * n) cap <<= 1;
    size_t head = (size_t)cap * 4 + 3 * n * 4 + 64;  // [slots cap][rep n][tid n][replist n][counter]
    if (head > ctx->dd_cap) {
        CK(cudaDeviceSynchronize());
        size_t want = ctx->dd_cap ? ctx->dd_cap : (1u << 20);
        while (want < head) want *= 2;
        cudaFree(ctx->dd_buf); ctx->dd_buf = nullptr; ctx->dd_cap = 0;
        CK(cudaMalloc(&ctx->dd_buf, want));
        ctx->dd_cap = want;
    }
    u32* slots = reinterpret_cast<u32*>(ctx->dd_buf);
    u32 *rep = slots + cap, *tid = rep + n, *replist = tid + n, *counter = replist + n;
    CK(cudaMemsetAsync(slots, 0xFF, (size_t)cap * 4, st));
    CK(cudaMemsetAsync(counter, 0, 4, st));
    unsigned gb = (unsigned)((n + 255) / 256);
    k_dedup_insert<<<gb, 256, 0, st>>>(d_key, keylen, n, slots, cap - 1, rep);
    k_dedup_number<<<gb, 256, 0, st>>>(rep, n, counter, tid, replist);
    k_dedup_resolve<<<gb, 256, 0, st>>>(rep, n, tid);
    ctx->launches += 3;
    u32 distinct = 0;
    CK(cudaMemcpyAsync(&distinct, counter, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (distinct_out) *distinct_out = distinct;
    if ((size_t)distinct * 10 > n * 6) return 0;  // fewer than 40 % repeats: the per-thread tables are as cheap
    size_t need_sk = (size_t)distinct * sizeof(sv_shared_key);
    if (need_sk > ctx->sk_cap) {
        CK(cudaDeviceSynchronize());
        size_t want = ctx->sk_cap ? ctx->sk_cap : (1u << 20);
        while (want < need_sk) want *= 2;
        cudaFree(ctx->sk_buf); ctx->sk_buf = nullptr; ctx->sk_cap = 0;
        CK(cudaMalloc(&ctx->sk_buf, want));
        ctx->sk_cap = want;
    }
    sv_shared_key* sk = reinterpret_cast<sv_shared_key*>(ctx->sk_buf);
    sv_ctx::slot_t* sl = nullptr;
    int rc = acquire_slot(ctx, n, st, &sl);
    if (rc) return rc;
    if (ctx->profiling) cudaEventRecord(ctx->ev[0], st);
    size_t threads = (n + SV_PREP_BATCH - 1) / SV_PREP_BATCH;
    k_prep_inv<<<(unsigned)((threads + 63) / 64), 64, 0, st>>>(d_msg, d_sig, n, sl->d_work);
    k_prep_finish<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(d_msg, d_sig, n, sl->d_work);
    if (ctx->profiling) cudaEventRecord(ctx->ev[1], st);
    k_sharedkey_build_many<<<(distinct + 127) / 128, 128, 0, st>>>(kind, d_key, keylen, replist, distinct, sk);
    size_t want = (n + SV_MAIN_BLOCK - 1) / SV_MAIN_BLOCK;
    unsigned grid = (unsigned)(want < (size_t)ctx->main_grid ? want : (size_t)ctx->main_grid);
    k_main_shared<<<grid, SV_MAIN_BLOCK, 0, st>>>(sl->d_work, d_sig, n, ctx->d_gtab, sk, tid, d_verdict, d_aux);
    if (ctx->profiling) cudaEventRecord(ctx->ev[2], st);
    ctx->launches += 4;
    CK(cudaGetLastError());
    rc = release_slot(ctx, sl, st);
    return rc ? rc : 1;
}

// L2 residency: the curve kernel re-reads the G comb table (34 MiB) and its own per-thread multiples tables (58 MiB per
// launch slot) ~70 times per verification, while inputs, work records and verdicts stream through once.  Round 1's ncu
// capture showed the slabs cycling through L2 to DRAM (1.33 GB per 1M launch, 10x the algorithmic bytes).  The window
// marks [G table | slabs] as persisting (as many of its lines as the carve-out holds) and everything else on the stream
// as streaming.
static void apply_l2_policy(sv_ctx* ctx, cudaStream_t st, const void* slab) {
    if (!ctx->l2_policy || !ctx->l2_persist) return;
    // one window per stream: the table slab of the launch slot this stream is about to use (58 MiB, written once and re-read
    // ~70 times per verification) plus the G comb table next to it (34 MiB): marked persisting they stay in L2 while inputs,
    // work records and verdicts stream past.  Measured (ncu, 1 M launch): slab-only window DRAM writes 728 -> 75 MB.  (A first attempt with one window over G table + both slabs at hit ratio carve-out/window RAISED the DRAM
    // traffic of a 1 M launch from 1.33 to 1.90 GB: the lines that lost the draw were treated as streaming.)
    for (int i = 0; i < 4; i++)
        if (ctx->policy_streams[i] == st && ctx->policy_slabs[i] == slab) return;
    cudaStreamAttrValue v;
    memset(&v, 0, sizeof v);
    // slot 0: [slab 0 | G table], slot 1: [G table | slab 1] — the slab and the comb table, the two things a verification re-reads
    const bool first = slab == (const void*)ctx->slot[0].d_scratch;
    v.accessPolicyWindow.base_ptr = first ? (void*)ctx->d_hot : (void*)ctx->d_gtab;
    v.accessPolicyWindow.num_bytes = ctx->hot_slab + ctx->hot_gt;
    double ratio = 0.95 * (double)ctx->l2_persist / (double)(ctx->hot_slab + ctx->hot_gt);
    v.accessPolicyWindow.hitRatio = (float)(ratio > 1.0 ? 1.0 : ratio);
    v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    v.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
    if (cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess) { (void)cudaGetLastError(); return; }
    for (int i = 3; i > 0; i--) { ctx->policy_streams[i] = ctx->policy_streams[i - 1]; ctx->policy_slabs[i] = ctx->policy_slabs[i - 1]; }
    ctx->policy_streams[0] = st;
    ctx->policy_slabs[0] = slab;
}

static int launch_small(sv_ctx* ctx, int kind, const u8* d_msg, const u8* d_key, const u8* d_sig, size_t n,
                        u8* d_verdict, u8* d_aux, cudaStream_t st) {
    unsigned grid = (unsigned)((n + SV_SMALL_ITEMS - 1) / SV_SMALL_ITEMS);
    if (ctx->profiling) cudaEventRecord(ctx->ev[0], st);
    if (ctx->profiling) cudaEventRecord(ctx->ev[1], st);
    // x-only keys: without the square root unless switched off (verify.cuh).  BIP-340 needs a field inversion at the end
    // either way, so dropping the square root is pure gain (n = 1: 471 -> 423 us).  For compressed-key ECDSA the division
    // D/B would be an inversion the plain flow does not have, as long as the square root it replaces and divergent across
    // lanes: measured slower (n = 32: 430 -> 529 us, profiles/r2_latency_small_nosqrt.json), so kind 0 stays on the plain flow.
    if (kind == SV_KIND_ECDSA33) k_small<SV_KIND_ECDSA33, false><<<grid, 160, 0, st>>>(d_msg, d_key, d_sig, n, ctx->d_gtab, d_verdict, d_aux);
    else if (kind == SV_KIND_ECDSA_XY) k_small<SV_KIND_ECDSA_XY, false><<<grid, 160, 0, st>>>(d_msg, d_key, d_sig, n, ctx->d_gtab, d_verdict, d_aux);
    else if (ctx->nosqrt) k_small<SV_KIND_SCHNORR, true><<<grid, 160, 0, st>>>(d_msg, d_key, d_sig, n, ctx->d_gtab, d_verdict, d_aux);
    else k_small<SV_KIND_SCHNORR, false><<<grid, 160, 0, st>>>(d_msg, d_key, d_sig, n, ctx->d_gtab, d_verdict, d_aux);
    if (ctx->profiling) cudaEventRecord(ctx->ev[2], st);
    ctx->launches += 1;
    CK(cudaGetLastError());
    return SV_OK;
}

static int launch_verify(sv_ctx* ctx, int kind, const u8* d_msg, const u8* d_key, const u8* d_sig, size_t n,
                         u8* d_verdict, u32* d_bitmap, cudaStream_t st, u8* d_keyok = nullptr) {
    if (n == 0) return SV_OK;
    if (n <= ctx->small_max) {  // few signatures: the latency-oriented kernel (one launch, three warps per verification)
        int rc = launch_small(ctx, kind, d_msg, d_key, d_sig, n, d_verdict, d_keyok, st);
        if (rc) return rc;
        if (d_bitmap) {
            k_pack_bitmap<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_verdict, n, d_bitmap);
            ctx->launches += 1;
            CK(cudaGetLastError());
        }
        return SV_OK;
    }
    sv_ctx::slot_t* sl = nullptr;
    int rc = acquire_slot(ctx, n, st, &sl);
    if (rc) return rc;
    apply_l2_policy(ctx, st, sl->d_scratch);
    sv_work* work = sl->d_work;
    if (ctx->profiling) cudaEventRecord(ctx->ev[0], st);
    if (kind == SV_KIND_SCHNORR) {
        k_prep_schnorr<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(d_msg, d_key, d_sig, n, work);
    } else {
        size_t threads = (n + SV_PREP_BATCH - 1) / SV_PREP_BATCH;
        k_prep_inv<<<(unsigned)((threads + 63) / 64), 64, 0, st>>>(d_msg, d_sig, n, work);
        k_prep_finish<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(d_msg, d_sig, n, work);
        ctx->launches += 1;
    }
    if (ctx->profiling) cudaEventRecord(ctx->ev[1], st);
    size_t want = (n + SV_MAIN_BLOCK - 1) / SV_MAIN_BLOCK;
    unsigned grid = (unsigned)(want < (size_t)ctx->main_grid ? want : (size_t)ctx->main_grid);
    if (kind == SV_KIND_ECDSA33 && ctx->nosqrt) {
        // compressed keys: the flow that skips the square root (verify.cuh "without the square root")
        k_main<SV_KIND_ECDSA33_NS><<<grid, SV_MAIN_BLOCK, SV_MAIN_SMEM, st>>>(work, d_key, d_sig, n, ctx->d_gtab, sl->d_scratch, d_verdict, nullptr);
        size_t threads = (n + SV_FINAL_BATCH - 1) / SV_FINAL_BATCH;
        k_final_ecdsa33<<<(unsigned)((threads + 63) / 64), 64, 0, st>>>(work, d_key, d_sig, n, ctx->d_gtab, d_verdict, d_keyok);
        ctx->launches += 1;
    } else if (kind == SV_KIND_ECDSA33)
        k_main<SV_KIND_ECDSA33><<<grid, SV_MAIN_BLOCK, SV_MAIN_SMEM, st>>>(work, d_key, d_sig, n, ctx->d_gtab, sl->d_scratch, d_verdict, d_keyok);
    else if (kind == SV_KIND_ECDSA_XY)
        k_main<SV_KIND_ECDSA_XY><<<grid, SV_MAIN_BLOCK, SV_MAIN_SMEM, st>>>(work, d_key, d_sig, n, ctx->d_gtab, sl->d_scratch, d_verdict, d_keyok);
    else if (ctx->nosqrt) {
        k_main<SV_KIND_SCHNORR_NS><<<grid, SV_MAIN_BLOCK, SV_MAIN_SMEM, st>>>(work, d_key, d_sig, n, ctx->d_gtab, sl->d_scratch, d_verdict, nullptr);
        size_t threads = (n + SV_FINAL_BATCH - 1) / SV_FINAL_BATCH;
        k_final_schnorr_ns<<<(unsigned)((threads + 63) / 64), 64, 0, st>>>(work, d_key, d_sig, n, ctx->d_gtab, d_verdict);
        ctx->launches += 1;
    } else {
        k_main<SV_KIND_SCHNORR><<<grid, SV_MAIN_BLOCK, SV_MAIN_SMEM, st>>>(work, d_key, d_sig, n, ctx->d_gtab, sl->d_scratch, d_verdict, d_keyok);
        size_t threads = (n + SV_FINAL_BATCH - 1) / SV_FINAL_BATCH;
        k_final_schnorr<<<(unsigned)((threads + 63) / 64), 64, 0, st>>>(work, d_sig, n, d_verdict);
        ctx->launches += 1;
    }
    if (ctx->profiling) cudaEventRecord(ctx->ev[2], st);
    ctx->launches += 2;
    if (d_bitmap) {
        size_t nb = (n + 255) / 256;
        k_pack_bitmap<<<(unsigned)nb, 256, 0, st>>>(d_verdict, n, d_bitmap);
        ctx->launches += 1;
    }
    CK(cudaGetLastError());
    return release_slot(ctx, sl, st);
}

extern "C" int sv_verify_device(sv_ctx* ctx, int kind, const void* d_msg32, const void* d_key, const void* d_sig64,
                                size_t n, void* d_verdicts, void* d_bitmap, void* stream) {
    if (!ctx || sv_key_size(kind) == 0 || (n && (!d_msg32 || !d_key || !d_sig64 || !d_verdicts))) return SV_ERR_ARG;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    return launch_verify(ctx, kind, (const u8*)d_msg32, (const u8*)d_key, (const u8*)d_sig64, n, (u8*)d_verdicts,
                         (u32*)d_bitmap, st);
}

extern "C" int sv_set_l2_policy(sv_ctx* ctx, int on) {
    if (!ctx) return SV_ERR_ARG;
    ctx->l2_policy = on ? 1 : 0;
    return SV_OK;
}
extern "C" int sv_set_dedup(sv_ctx* ctx, int on) {
    if (!ctx) return SV_ERR_ARG;
    ctx->dedup = on ? 1 : 0;
    return SV_OK;
}
extern "C" int sv_set_nosqrt(sv_ctx* ctx, int on) {
    if (!ctx) return SV_ERR_ARG;
    ctx->nosqrt = on ? 1 : 0;
    return SV_OK;
}
extern "C" unsigned sv_last_distinct_keys(const sv_ctx* ctx) { return ctx ? ctx->last_distinct : 0; }
extern "C" int sv_set_small_max(sv_ctx* ctx, size_t n) {
    if (!ctx) return SV_ERR_ARG;
    ctx->small_max = n < ctx->small_cap ? n : ctx->small_cap;
    return SV_OK;
}
extern "C" size_t sv_get_small_max(const sv_ctx* ctx) { return ctx ? ctx->small_max : 0; }

extern "C" int sv_set_profiling(sv_ctx* ctx, int on) {
    if (!ctx) return SV_ERR_ARG;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    if (on && !ctx->ev[0])
        for (int i = 0; i < 3; i++) CK(cudaEventCreate(&ctx->ev[i]));
    ctx->profiling = on ? 1 : 0;
    return SV_OK;
}
// device time of the last sv_verify_* launch pair (call after the stream has been synchronised)
extern "C" int sv_get_last_timing(sv_ctx* ctx, float* prep_ms, float* main_ms) {
    if (!ctx || !ctx->profiling || !prep_ms || !main_ms) return SV_ERR_ARG;
    CK(cudaEventElapsedTime(prep_ms, ctx->ev[0], ctx->ev[1]));
    CK(cudaEventElapsedTime(main_ms, ctx->ev[1], ctx->ev[2]));
    return SV_OK;
}

extern "C" void* sv_get_stream(const sv_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

extern "C" int sv_sync(sv_ctx* ctx, void* stream) {
    if (!ctx) return SV_ERR_ARG;
    CK(cudaStreamSynchronize(stream ? (cudaStream_t)stream : ctx->stream));
    return SV_OK;
}

#ifndef SV_HOST_CHUNK
#define SV_HOST_CHUNK (1u << 21)
#endif

extern "C" int sv_verify_host(sv_ctx* ctx, int kind, const uint8_t* msg32, const uint8_t* key, const uint8_t* sig64,
                              size_t n, uint8_t* verdicts) {
    size_t ks_ = sv_key_size(kind);
    if (!ctx || ks_ == 0 || (n && (!msg32 || !key || !sig64 || !verdicts))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    if (n <= ctx->small_max) {
        // small batch: inputs go through the pinned staging block, the kernel reads them over the bus itself and writes the
        // verdict bytes back the same way: one launch and one stream synchronisation, nothing else
        u8 *hm = ctx->h_small, *hk = hm + 32 * ctx->small_cap, *hs = hk + 64 * ctx->small_cap, *hv = hs + 64 * ctx->small_cap;
        memcpy(hm, msg32, 32 * n);
        memcpy(hk, key, ks_ * n);
        memcpy(hs, sig64, 64 * n);
        int rc = launch_small(ctx, kind, hm, hk, hs, n, hv, nullptr, ctx->stream);
        if (rc) return rc;
        CK(cudaStreamSynchronize(ctx->stream));
        memcpy(verdicts, hv, n);
        return SV_OK;
    }
    size_t chunk = n < SV_HOST_CHUNK ? n : SV_HOST_CHUNK;
    int rc = ensure_staging(ctx, chunk);
    if (rc) return rc;
    // Software pipeline inside a chunk: slices sized in whole waves of the persistent grid; slice k+1 is copied on
    // the copy stream while slice k runs; consecutive slices alternate between the two compute streams (each has its own
    // launch slot), so the partially filled last wave of one slice overlaps the next slice.  First slice small so the
    // kernels start early — and it also takes the odd remainder of the chunk: its thin last wave is covered by the second
    // slice, and the LAST slice (whose tail nothing can cover: the call is synchronous) ends on a full wave.
    const size_t wave = (size_t)ctx->main_grid * SV_MAIN_BLOCK;
    for (size_t off = 0; off < n; off += chunk) {
        size_t c = (n - off < chunk) ? (n - off) : chunk;
        size_t done = 0;
        int k = 0;
        const bool piped = c > 2 * wave;
        while (done < c) {
            size_t want = (k == 0) ? wave + c % wave : 6 * wave;
            size_t s = (c - done <= want + 2 * wave) ? (c - done) : want;  // do not leave a sliver behind
            if (k >= 7) s = c - done;
            cudaStream_t cs = piped ? ctx->copy_stream : ctx->stream;
            cudaStream_t ks = (piped && (k & 1)) ? ctx->stream2 : ctx->stream;
            CK(cudaMemcpyAsync(ctx->d_msg + 32 * done, msg32 + 32 * (off + done), 32 * s, cudaMemcpyHostToDevice, cs));
            CK(cudaMemcpyAsync(ctx->d_key + ks_ * done, key + ks_ * (off + done), ks_ * s, cudaMemcpyHostToDevice, cs));
            CK(cudaMemcpyAsync(ctx->d_sig + 64 * done, sig64 + 64 * (off + done), 64 * s, cudaMemcpyHostToDevice, cs));
            if (cs != ks) {
                CK(cudaEventRecord(ctx->h2d_ev[k], cs));
                CK(cudaStreamWaitEvent(ks, ctx->h2d_ev[k], 0));
            }
            rc = launch_verify(ctx, kind, ctx->d_msg + 32 * done, ctx->d_key + ks_ * done, ctx->d_sig + 64 * done, s,
                               ctx->d_verdict + done, nullptr, ks);
            if (rc) return rc;
            CK(cudaMemcpyAsync(verdicts + off + done, ctx->d_verdict + done, s, cudaMemcpyDeviceToHost, ks));
            done += s;
            k++;
        }
        // the next chunk reuses the staging buffers: its copies must not overtake this chunk's kernels
        CK(cudaStreamSynchronize(ctx->stream));
        if (piped) CK(cudaStreamSynchronize(ctx->stream2));
    }
    return SV_OK;
}

static int stage_spans(sv_ctx* ctx, const uint8_t* data, size_t data_len, const uint64_t* off, const uint32_t* len,
                       size_t n) {
    for (size_t i = 0; i < n; i++)
        if (off[i] > data_len || (size_t)len[i] > data_len - off[i]) return fail(ctx, SV_ERR_ARG, "span out of range", cudaSuccess);
    if (data_len > ctx->data_cap) {
        cudaFree(ctx->d_data); ctx->d_data = nullptr; ctx->data_cap = 0;
        CK(cudaMalloc(&ctx->d_data, data_len ? data_len : 1));
        ctx->data_cap = data_len;
    }
    if (n > ctx->span_cap) {
        cudaFree(ctx->d_off); cudaFree(ctx->d_len); ctx->d_off = nullptr; ctx->d_len = nullptr; ctx->span_cap = 0;
        CK(cudaMalloc(&ctx->d_off, n * sizeof(u64)));
        CK(cudaMalloc(&ctx->d_len, n * sizeof(u32)));
        ctx->span_cap = n;
    }
    CK(cudaMemcpyAsync(ctx->d_data, data, data_len, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_off, off, n * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_len, len, n * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    return SV_OK;
}

extern "C" int sv_verify_host_raw(sv_ctx* ctx, int kind, const uint8_t* data, size_t data_len, const uint64_t* off,
                                  const uint32_t* len, const uint8_t* key, const uint8_t* sig64, size_t n,
                                  uint8_t* verdicts) {
    size_t ks = sv_key_size(kind);
    if (!ctx || ks == 0 || (n && (!data || !off || !len || !key || !sig64 || !verdicts))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    int rc = ensure_staging(ctx, n);
    if (rc) return rc;
    rc = stage_spans(ctx, data, data_len, off, len, n);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->d_key, key, ks * n, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_sig, sig64, 64 * n, cudaMemcpyHostToDevice, ctx->stream));
    k_sha256d<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(ctx->d_data, ctx->d_off, ctx->d_len, n, ctx->d_msg);
    ctx->launches += 1;
    rc = launch_verify(ctx, kind, ctx->d_msg, ctx->d_key, ctx->d_sig, n, ctx->d_verdict, nullptr, ctx->stream);
    if (rc) return rc;
    CK(cudaMemcpyAsync(verdicts, ctx->d_verdict, n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SV_OK;
}

extern "C" int sv_sha256d_host(sv_ctx* ctx, const uint8_t* data, size_t data_len, const uint64_t* off,
                               const uint32_t* len, size_t n, uint8_t* out32) {
    if (!ctx || (n && (!data || !off || !len || !out32))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    int rc = ensure_staging(ctx, n);
    if (rc) return rc;
    rc = stage_spans(ctx, data, data_len, off, len, n);
    if (rc) return rc;
    k_sha256d<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(ctx->d_data, ctx->d_off, ctx->d_len, n, ctx->d_msg);
    ctx->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out32, ctx->d_msg, 32 * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SV_OK;
}

extern "C" int sv_pubkey_parse_host(sv_ctx* ctx, const uint8_t* key33, size_t n, uint8_t* xy64, uint8_t* ok) {
    if (!ctx || (n && (!key33 || !xy64 || !ok))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    int rc = ensure_staging(ctx, n);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->d_key, key33, 33 * n, cudaMemcpyHostToDevice, ctx->stream));
    k_pubkey_parse<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(ctx->d_key, n, ctx->d_sig, ctx->d_verdict);
    ctx->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(xy64, ctx->d_sig, 64 * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ok, ctx->d_verdict, n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SV_OK;
}

// gossip ingest with device-side slicing: blob = concatenated wire messages, msg_off/msg_len locate them.
extern "C" int sv_verify_gossip_host(sv_ctx* ctx, const uint8_t* blob, size_t blob_len, const uint64_t* msg_off,
                                     const uint32_t* msg_len, size_t n_msgs, const uint8_t* cu_signers33, int* status) {
    if (!ctx || (n_msgs && (!blob || !msg_off || !msg_len || !status))) return SV_ERR_ARG;
    if (n_msgs == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    // the host only reads the 2-byte type of each message to lay out the item slots
    std::vector<u32> base(n_msgs);
    size_t items = 0;
    for (size_t m = 0; m < n_msgs; m++) {
        if (msg_off[m] > blob_len || msg_len[m] > blob_len - msg_off[m]) return fail(ctx, SV_ERR_ARG, "message out of range", cudaSuccess);
        u32 type = msg_len[m] >= 2 ? (((u32)blob[msg_off[m]] << 8) | blob[msg_off[m] + 1]) : 0;
        base[m] = (u32)items;
        items += (type == 256) ? 4 : ((type == 257 || type == 258) ? 1 : 0);
    }
    size_t cap = items ? items : 1;
    int rc = ensure_staging(ctx, cap);
    if (rc) return rc;
    if (blob_len > ctx->data_cap) {
        cudaFree(ctx->d_data); ctx->d_data = nullptr; ctx->data_cap = 0;
        CK(cudaMalloc(&ctx->d_data, blob_len));
        ctx->data_cap = blob_len;
    }
    size_t need = (cap > n_msgs ? cap : n_msgs);
    if (need > ctx->span_cap) {
        cudaFree(ctx->d_off); cudaFree(ctx->d_len); ctx->d_off = nullptr; ctx->d_len = nullptr; ctx->span_cap = 0;
        CK(cudaMalloc(&ctx->d_off, need * sizeof(u64)));
        CK(cudaMalloc(&ctx->d_len, need * sizeof(u32)));
        ctx->span_cap = need;
    }
    // one grow-only slab: [msg_off u64][msg_len u32][item_base u32][status int][signers 33B][keyok 1B per item]
    size_t need_g = n_msgs * (8 + 4 + 4 + 4 + 33) + cap + 64;
    if (need_g > ctx->g_cap) {
        CK(cudaDeviceSynchronize());
        size_t gcap = ctx->g_cap ? ctx->g_cap : (1u << 16);
        while (gcap < need_g) gcap *= 2;
        cudaFree(ctx->g_buf); ctx->g_buf = nullptr; ctx->g_cap = 0;
        CK(cudaMalloc(&ctx->g_buf, gcap));
        ctx->g_cap = gcap;
    }
    u64* d_moff = reinterpret_cast<u64*>(ctx->g_buf);
    u32* d_mlen = reinterpret_cast<u32*>(d_moff + n_msgs);
    u32* d_base = d_mlen + n_msgs;
    int* d_status = reinterpret_cast<int*>(d_base + n_msgs);
    u8* d_signers = reinterpret_cast<u8*>(d_status + n_msgs);
    u8* d_keyok = d_signers + 33 * n_msgs;
    if (!cu_signers33) d_signers = nullptr;
    cudaStream_t st = ctx->stream;
    CK(cudaMemcpyAsync(ctx->d_data, blob, blob_len, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_moff, msg_off, n_msgs * sizeof(u64), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_mlen, msg_len, n_msgs * sizeof(u32), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_base, base.data(), n_msgs * sizeof(u32), cudaMemcpyHostToDevice, st));
    if (cu_signers33) CK(cudaMemcpyAsync(d_signers, cu_signers33, n_msgs * 33, cudaMemcpyHostToDevice, st));
    unsigned gm = (unsigned)((n_msgs + 127) / 128);
    k_gossip_slice<<<gm, 128, 0, st>>>(ctx->d_data, d_moff, d_mlen, d_base, d_signers, n_msgs, ctx->d_off, ctx->d_len,
                                       ctx->d_key, ctx->d_sig, d_status);
    ctx->launches += 1;
    if (items) {
        k_sha256d<<<(unsigned)((items + 127) / 128), 128, 0, st>>>(ctx->d_data, ctx->d_off, ctx->d_len, items, ctx->d_msg);
        ctx->launches += 1;
        // node keys repeat heavily inside a gossip batch (every channel of a node, its updates, its announcement)
        rc = ctx->dedup ? launch_verify_dedup(ctx, SV_KIND_ECDSA33, ctx->d_msg, ctx->d_key, ctx->d_sig, items, ctx->d_verdict, st, d_keyok,
                                              &ctx->last_distinct) : 0;
        if (rc == 0) rc = launch_verify(ctx, SV_KIND_ECDSA33, ctx->d_msg, ctx->d_key, ctx->d_sig, items, ctx->d_verdict, nullptr, st, d_keyok);
        else if (rc == 1) rc = SV_OK;
        if (rc == SV_OK) {
            k_gossip_status<<<gm, 128, 0, st>>>(ctx->d_data, d_moff, d_mlen, d_base, n_msgs, ctx->d_verdict, d_keyok, d_status);
            ctx->launches += 1;
        }
    }
    cudaError_t ce = cudaMemcpyAsync(status, d_status, n_msgs * sizeof(int), cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
    if (rc) return rc;
    if (ce != cudaSuccess) return fail(ctx, SV_ERR_CUDA, "gossip ingest", ce);
    return SV_OK;
}

// n ECDSA signatures by ONE key (channeld's HTLC loop): table of the key built once, ladder-only kernel
extern "C" int sv_verify_samekey_host(sv_ctx* ctx, int kind, const uint8_t* key, const uint8_t* msg32, const uint8_t* sig64,
                                      size_t n, uint8_t* verdicts) {
    size_t ks = sv_key_size(kind);
    if (!ctx || ks == 0 || kind == SV_KIND_SCHNORR || (n && (!key || !msg32 || !sig64 || !verdicts))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    if (n <= ctx->small_max) {
        // a commitment_signed carries at most 483 HTLC signatures: latency matters more than the 18 % of work a shared
        // table saves, so small same-key batches take the small-batch path with the key repeated per item
        u8 *hm = ctx->h_small, *hk = hm + 32 * ctx->small_cap, *hs = hk + 64 * ctx->small_cap, *hv = hs + 64 * ctx->small_cap;
        memcpy(hm, msg32, 32 * n);
        for (size_t i = 0; i < n; i++) memcpy(hk + ks * i, key, ks);
        memcpy(hs, sig64, 64 * n);
        int rcs = launch_small(ctx, kind, hm, hk, hs, n, hv, nullptr, ctx->stream);
        if (rcs) return rcs;
        CK(cudaStreamSynchronize(ctx->stream));
        memcpy(verdicts, hv, n);
        return SV_OK;
    }
    int rc = ensure_staging(ctx, n);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    sv_ctx::slot_t* sl = nullptr;
    rc = acquire_slot(ctx, n, st, &sl);
    if (rc) return rc;
    // the shared key's table lives at the head of the slot's (otherwise unused) per-thread table slab
    sv_shared_key* d_sk = reinterpret_cast<sv_shared_key*>(sl->d_scratch);
    CK(cudaMemcpyAsync(ctx->d_key, key, ks, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_msg, msg32, 32 * n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_sig, sig64, 64 * n, cudaMemcpyHostToDevice, st));
    k_sharedkey_build<<<1, 32, 0, st>>>(kind, ctx->d_key, d_sk);
    size_t threads = (n + SV_PREP_BATCH - 1) / SV_PREP_BATCH;
    k_prep_inv<<<(unsigned)((threads + 63) / 64), 64, 0, st>>>(ctx->d_msg, ctx->d_sig, n, sl->d_work);
    k_prep_finish<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(ctx->d_msg, ctx->d_sig, n, sl->d_work);
    ctx->launches += 1;
    size_t want = (n + SV_MAIN_BLOCK - 1) / SV_MAIN_BLOCK;
    unsigned grid = (unsigned)(want < (size_t)ctx->main_grid ? want : (size_t)ctx->main_grid);
    k_main_shared<<<grid, SV_MAIN_BLOCK, 0, st>>>(sl->d_work, ctx->d_sig, n, ctx->d_gtab, d_sk, nullptr, ctx->d_verdict, nullptr);
    ctx->launches += 3;
    cudaError_t ce = cudaGetLastError();
    if (ce == cudaSuccess) ce = cudaEventRecord(sl->done, st);
    sl->last_stream = st;
    sl->used = 1;
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(verdicts, ctx->d_verdict, n, cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
    if (ce != cudaSuccess) return fail(ctx, SV_ERR_CUDA, "sv_verify_samekey_host", ce);
    return SV_OK;
}

// check_tx_sig with the BIP143 sighash computed on the device (channeld's per-HTLC loop as one launch)
static_assert(sizeof(sv_tx_item) == sizeof(sv_tx), "host and device views of the transaction item must agree");
extern "C" int sv_verify_tx_host(sv_ctx* ctx, int kind, const sv_tx* txs, const uint8_t* scripts, size_t scripts_len,
                                 const uint8_t* key, const uint8_t* sig64, size_t n, uint8_t* verdicts,
                                 uint8_t* sighash32_out) {
    size_t ks = sv_key_size(kind);
    if (!ctx || ks == 0 || kind == SV_KIND_SCHNORR || (n && (!txs || !key || !sig64 || !verdicts))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    for (size_t i = 0; i < n; i++)
        if ((size_t)txs[i].script_off + txs[i].script_len > scripts_len ||
            (size_t)txs[i].out_script_off + txs[i].out_script_len > scripts_len ||
            ((txs[i].flags & SV_TX_INPUTS_SERIALIZED) &&
             ((size_t)txs[i].prevouts_off + txs[i].prevouts_len > scripts_len ||
              (size_t)txs[i].sequences_off + txs[i].sequences_len > scripts_len)))
            return fail(ctx, SV_ERR_ARG, "script span out of range", cudaSuccess);
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    int rc = ensure_staging(ctx, n);
    if (rc) return rc;
    if (scripts_len + 1 > ctx->data_cap) {
        cudaFree(ctx->d_data); ctx->d_data = nullptr; ctx->data_cap = 0;
        CK(cudaMalloc(&ctx->d_data, scripts_len + 1));
        ctx->data_cap = scripts_len + 1;
    }
    // transaction records + sighash-ok flags in the grow-only auxiliary slab (no allocation on the steady-state call path)
    size_t need_g = n * sizeof(sv_tx_item) + n + 64;
    if (need_g > ctx->g_cap) {
        CK(cudaDeviceSynchronize());
        size_t cap = ctx->g_cap ? ctx->g_cap : (1u << 16);
        while (cap < need_g) cap *= 2;
        cudaFree(ctx->g_buf); ctx->g_buf = nullptr; ctx->g_cap = 0;
        CK(cudaMalloc(&ctx->g_buf, cap));
        ctx->g_cap = cap;
    }
    sv_tx_item* d_txs = reinterpret_cast<sv_tx_item*>(ctx->g_buf);
    u8* d_ok = ctx->g_buf + n * sizeof(sv_tx_item);
    cudaStream_t st = ctx->stream;
    CK(cudaMemcpyAsync(d_txs, txs, n * sizeof(sv_tx_item), cudaMemcpyHostToDevice, st));
    if (scripts_len) CK(cudaMemcpyAsync(ctx->d_data, scripts, scripts_len, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_key, key, ks * n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_sig, sig64, 64 * n, cudaMemcpyHostToDevice, st));
    k_bip143<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(d_txs, ctx->d_data, n, ctx->d_msg, d_ok);
    ctx->launches += 1;
    rc = launch_verify(ctx, kind, ctx->d_msg, ctx->d_key, ctx->d_sig, n, ctx->d_verdict, nullptr, st);
    cudaError_t ce = cudaSuccess;
    if (rc == SV_OK) {
        k_mask_verdicts<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ctx->d_verdict, d_ok, n);
        ctx->launches += 1;
        ce = cudaMemcpyAsync(verdicts, ctx->d_verdict, n, cudaMemcpyDeviceToHost, st);
        if (ce == cudaSuccess && sighash32_out) ce = cudaMemcpyAsync(sighash32_out, ctx->d_msg, 32 * n, cudaMemcpyDeviceToHost, st);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
    }
    if (rc) return rc;
    if (ce != cudaSuccess) return fail(ctx, SV_ERR_CUDA, "sv_verify_tx_host", ce);
    return SV_OK;
}

// ---- mixed batches: kinds[n] tags, keys in 64-byte slots (the first 33 / 64 / 32 bytes used) ----------------------
static int ensure_gbuf(sv_ctx* ctx, size_t need) {
    if (need <= ctx->g_cap) return SV_OK;
    CK(cudaDeviceSynchronize());
    size_t cap = ctx->g_cap ? ctx->g_cap : (1u << 16);
    while (cap < need) cap *= 2;
    cudaFree(ctx->g_buf); ctx->g_buf = nullptr; ctx->g_cap = 0;
    CK(cudaMalloc(&ctx->g_buf, cap));
    ctx->g_cap = cap;
    return SV_OK;
}
// inputs already on the device; scratch = [count u32 x4][idx u32 x 3n]; staging = the context's SoA staging arrays
static int mixed_device(sv_ctx* ctx, const u8* d_kinds, const u8* d_msg, const u8* d_key64, const u8* d_sig, size_t n,
                        u8* d_out, u32* d_scratch, cudaStream_t st) {
    u32* d_count = d_scratch;
    u32* d_idx = d_scratch + 4;
    CK(cudaMemsetAsync(d_count, 0, 16, st));
    CK(cudaMemsetAsync(d_out, 0, n, st));
    k_mixed_index<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_kinds, n, d_count, d_idx);
    ctx->launches += 1;
    u32 count[4];
    CK(cudaMemcpyAsync(count, d_count, 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));  // the per-kind launch sizes are needed on the host
    size_t o = 0;
    for (int kind = 0; kind < 3; kind++) {
        size_t c = count[kind];
        if (!c) continue;
        size_t ks = sv_key_size(kind);
        u8 *om = ctx->d_msg + 32 * o, *ok = ctx->d_key + 64 * o, *os = ctx->d_sig + 64 * o, *ov = ctx->d_verdict + o;
        const u32* list = d_idx + (size_t)kind * n;
        k_mixed_gather<<<(unsigned)((c + 255) / 256), 256, 0, st>>>(list, c, (int)ks, d_msg, d_key64, d_sig, om, ok, os);
        int rc = launch_verify(ctx, kind, om, ok, os, c, ov, nullptr, st);
        if (rc) return rc;
        k_mixed_scatter<<<(unsigned)((c + 255) / 256), 256, 0, st>>>(list, c, ov, d_out);
        ctx->launches += 2;
        o += c;
    }
    CK(cudaGetLastError());
    return SV_OK;
}
extern "C" int sv_verify_mixed_device(sv_ctx* ctx, const void* d_kinds, const void* d_msg32, const void* d_key64,
                                      const void* d_sig64, size_t n, void* d_verdicts, void* stream) {
    if (!ctx || (n && (!d_kinds || !d_msg32 || !d_key64 || !d_sig64 || !d_verdicts))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    int rc = ensure_staging(ctx, n);
    if (rc) return rc;
    rc = ensure_gbuf(ctx, 16 + 12 * n + 64);
    if (rc) return rc;
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    return mixed_device(ctx, (const u8*)d_kinds, (const u8*)d_msg32, (const u8*)d_key64, (const u8*)d_sig64, n,
                        (u8*)d_verdicts, reinterpret_cast<u32*>(ctx->g_buf), st);
}
extern "C" int sv_verify_mixed_host(sv_ctx* ctx, const uint8_t* kinds, const uint8_t* msg32, const uint8_t* key64,
                                    const uint8_t* sig64, size_t n, uint8_t* verdicts) {
    if (!ctx || (n && (!kinds || !msg32 || !key64 || !sig64 || !verdicts))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    int rc = ensure_staging(ctx, n);
    if (rc) return rc;
    // aux slab: [count + idx lists][kinds n][msg 32n][key 64n][sig 64n][out n], 16-byte aligned pieces
    size_t a = (16 + 12 * n + 15) & ~(size_t)15, need = a + ((n + 15) & ~(size_t)15) * 2 + 160 * n + 64;
    rc = ensure_gbuf(ctx, need);
    if (rc) return rc;
    u8* d_kinds = ctx->g_buf + a;
    u8* d_m = d_kinds + ((n + 15) & ~(size_t)15);
    u8* d_k = d_m + 32 * n;
    u8* d_s = d_k + 64 * n;
    u8* d_o = d_s + 64 * n;
    cudaStream_t st = ctx->stream;
    CK(cudaMemcpyAsync(d_kinds, kinds, n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_m, msg32, 32 * n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_k, key64, 64 * n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_s, sig64, 64 * n, cudaMemcpyHostToDevice, st));
    rc = mixed_device(ctx, d_kinds, d_m, d_k, d_s, n, d_o, reinterpret_cast<u32*>(ctx->g_buf), st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(verdicts, d_o, n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SV_OK;
}

// ---- public-key recovery (secp256k1_ecdsa_recover; verify.cuh "public-key recovery") -----------------------------------
// inputs on the device: recid[n] bytes, keys to d_xy (64 bytes per item), status bytes (int8_t) to d_status
static int launch_recover(sv_ctx* ctx, const u8* d_msg, const u8* d_recid, const u8* d_sig, size_t n, u8* d_xy, u8* d_status,
                          cudaStream_t st) {
    if (n == 0) return SV_OK;
    if (n <= ctx->small_max) {
        unsigned grid = (unsigned)((n + SV_SMALL_ITEMS - 1) / SV_SMALL_ITEMS);
        if (ctx->profiling) cudaEventRecord(ctx->ev[0], st);
        if (ctx->profiling) cudaEventRecord(ctx->ev[1], st);
        k_small<SV_KIND_RECOVER, false><<<grid, 160, 0, st>>>(d_msg, d_recid, d_sig, n, ctx->d_gtab, d_status, d_xy);
        if (ctx->profiling) cudaEventRecord(ctx->ev[2], st);
        ctx->launches += 1;
        CK(cudaGetLastError());
        return SV_OK;
    }
    sv_ctx::slot_t* sl = nullptr;
    int rc = acquire_slot(ctx, n, st, &sl);
    if (rc) return rc;
    apply_l2_policy(ctx, st, sl->d_scratch);
    sv_work* work = sl->d_work;
    if (ctx->profiling) cudaEventRecord(ctx->ev[0], st);
    size_t threads = (n + SV_PREP_BATCH - 1) / SV_PREP_BATCH;
    k_prep_recover_inv<<<(unsigned)((threads + 63) / 64), 64, 0, st>>>(d_msg, d_sig, d_recid, n, work);
    k_prep_recover_finish<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(d_msg, d_sig, d_recid, n, work);
    if (ctx->profiling) cudaEventRecord(ctx->ev[1], st);
    size_t want = (n + SV_MAIN_BLOCK - 1) / SV_MAIN_BLOCK;
    unsigned grid = (unsigned)(want < (size_t)ctx->main_grid ? want : (size_t)ctx->main_grid);
    k_main<SV_KIND_RECOVER><<<grid, SV_MAIN_BLOCK, SV_MAIN_SMEM, st>>>(work, d_recid, d_sig, n, ctx->d_gtab, sl->d_scratch, nullptr, nullptr);
    threads = (n + SV_FINAL_BATCH - 1) / SV_FINAL_BATCH;
    k_final_recover<<<(unsigned)((threads + 63) / 64), 64, 0, st>>>(work, n, d_xy, d_status);
    if (ctx->profiling) cudaEventRecord(ctx->ev[2], st);
    ctx->launches += 4;
    CK(cudaGetLastError());
    return release_slot(ctx, sl, st);
}

extern "C" int sv_recover_host(sv_ctx* ctx, const uint8_t* msg32, const uint8_t* sig64, const uint8_t* recid, size_t n,
                               uint8_t* xy64, int8_t* status) {
    if (!ctx || (n && (!msg32 || !sig64 || !recid || !xy64 || !status))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    if (n <= ctx->small_max) {
        // pinned staging block as in sv_verify_host: recids in the second byte per item of the verdict area, keys come
        // back through the key area (the kernel never reads it for this kind)
        const size_t cap = ctx->small_cap;
        u8 *hm = ctx->h_small, *hk = hm + 32 * cap, *hs = hk + 64 * cap, *hv = hs + 64 * cap;
        memcpy(hm, msg32, 32 * n);
        memcpy(hv + cap, recid, n);
        memcpy(hs, sig64, 64 * n);
        int rc = launch_recover(ctx, hm, hv + cap, hs, n, hk, hv, ctx->stream);
        if (rc) return rc;
        CK(cudaStreamSynchronize(ctx->stream));
        memcpy(xy64, hk, 64 * n);
        memcpy(status, hv, n);
        return SV_OK;
    }
    size_t chunk = n < SV_HOST_CHUNK ? n : SV_HOST_CHUNK;
    int rc = ensure_staging(ctx, chunk);
    if (rc) return rc;
    rc = ensure_gbuf(ctx, 64 * chunk);  // the keys of one chunk
    if (rc) return rc;
    u8* d_xy = ctx->g_buf;
    // the slicing and stream pipeline of sv_verify_host; the recid bytes travel in the key staging array
    const size_t wave = (size_t)ctx->main_grid * SV_MAIN_BLOCK;
    for (size_t off = 0; off < n; off += chunk) {
        size_t c = (n - off < chunk) ? (n - off) : chunk;
        size_t done = 0;
        int k = 0;
        const bool piped = c > 2 * wave;
        while (done < c) {
            size_t want = (k == 0) ? wave + c % wave : 6 * wave;
            size_t s = (c - done <= want + 2 * wave) ? (c - done) : want;
            if (k >= 7) s = c - done;
            cudaStream_t cs = piped ? ctx->copy_stream : ctx->stream;
            cudaStream_t ks = (piped && (k & 1)) ? ctx->stream2 : ctx->stream;
            CK(cudaMemcpyAsync(ctx->d_msg + 32 * done, msg32 + 32 * (off + done), 32 * s, cudaMemcpyHostToDevice, cs));
            CK(cudaMemcpyAsync(ctx->d_key + done, recid + off + done, s, cudaMemcpyHostToDevice, cs));
            CK(cudaMemcpyAsync(ctx->d_sig + 64 * done, sig64 + 64 * (off + done), 64 * s, cudaMemcpyHostToDevice, cs));
            if (cs != ks) {
                CK(cudaEventRecord(ctx->h2d_ev[k], cs));
                CK(cudaStreamWaitEvent(ks, ctx->h2d_ev[k], 0));
            }
            rc = launch_recover(ctx, ctx->d_msg + 32 * done, ctx->d_key + done, ctx->d_sig + 64 * done, s, d_xy + 64 * done,
                                ctx->d_verdict + done, ks);
            if (rc) return rc;
            CK(cudaMemcpyAsync(xy64 + 64 * (off + done), d_xy + 64 * done, 64 * s, cudaMemcpyDeviceToHost, ks));
            CK(cudaMemcpyAsync(status + off + done, ctx->d_verdict + done, s, cudaMemcpyDeviceToHost, ks));
            done += s;
            k++;
        }
        CK(cudaStreamSynchronize(ctx->stream));
        if (piped) CK(cudaStreamSynchronize(ctx->stream2));
    }
    return SV_OK;
}

// ---- BIP-340 batch verification, host entry (batch.cuh) --------------------------------------------------------------
#include <sys/random.h>
extern "C" int sv_verify_schnorr_batch_host(sv_ctx* ctx, const uint8_t* msg32, const uint8_t* xonly32, const uint8_t* sig64,
                                            size_t n, const uint8_t* seed32, uint8_t* verdicts, uint32_t* groups_total,
                                            uint32_t* groups_failed) {
    if (!ctx || (n && (!msg32 || !xonly32 || !sig64 || !verdicts))) return SV_ERR_ARG;
    if (groups_total) *groups_total = 0;
    if (groups_failed) *groups_failed = 0;
    if (n == 0) return SV_OK;
    if (n > 0x7FFFFFFFu) return SV_ERR_ARG;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    uint8_t seed[32];
    if (seed32) memcpy(seed, seed32, 32);
    else if (getrandom(seed, 32, 0) != 32) return fail(ctx, SV_ERR_ARG, "getrandom", cudaSuccess);
    int rc = ensure_staging(ctx, n);
    if (rc) return rc;
    const u32 groups = (u32)((n + SV_SB_GROUP - 1) / SV_SB_GROUP);
    // scratch: [seed 32][pts 2n x 96][t n x 32][S groups x W x 128][dig W x 4n][ok n][group_ok groups][out n][idx n x 4]
    size_t o_pts = 64, o_t = o_pts + 2 * n * sizeof(qtab_entry), o_S = o_t + n * sizeof(sc),
           o_dig = o_S + (size_t)groups * SV_SB_WINDOWS * sizeof(sv_jac), o_ok = (o_dig + (size_t)SV_SB_WINDOWS * 4 * n + 15) & ~(size_t)15,
           o_gok = (o_ok + n + 15) & ~(size_t)15, o_out = (o_gok + groups + 15) & ~(size_t)15, o_idx = (o_out + n + 15) & ~(size_t)15,
           need = o_idx + 4 * n + 64;
    if (need > ctx->dd_cap) {
        CK(cudaDeviceSynchronize());
        size_t want = ctx->dd_cap ? ctx->dd_cap : (1u << 20);
        while (want < need) want *= 2;
        cudaFree(ctx->dd_buf); ctx->dd_buf = nullptr; ctx->dd_cap = 0;
        CK(cudaMalloc(&ctx->dd_buf, want));
        ctx->dd_cap = want;
    }
    u8* B = ctx->dd_buf;
    qtab_entry* d_pts = reinterpret_cast<qtab_entry*>(B + o_pts);
    sc* d_t = reinterpret_cast<sc*>(B + o_t);
    sv_jac* d_S = reinterpret_cast<sv_jac*>(B + o_S);
    signed char* d_dig = reinterpret_cast<signed char*>(B + o_dig);
    u8 *d_ok = B + o_ok, *d_gok = B + o_gok, *d_out = B + o_out;
    u32* d_idx = reinterpret_cast<u32*>(B + o_idx);
    cudaStream_t st = ctx->stream;
    CK(cudaMemcpyAsync(B, seed, 32, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_msg, msg32, 32 * n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_key, xonly32, 32 * n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_sig, sig64, 64 * n, cudaMemcpyHostToDevice, st));
    if (ctx->profiling) cudaEventRecord(ctx->ev[0], st);
    if (sv_batch_launch(ctx->d_msg, ctx->d_key, ctx->d_sig, n, B, d_pts, d_dig, d_t, d_ok, d_S, d_gok, d_out, ctx->d_gtab, st,
                        ctx->profiling ? ctx->ev[1] : nullptr) != 0)
        return fail(ctx, SV_ERR_CUDA, "batch kernels", cudaGetLastError());
    if (ctx->profiling) cudaEventRecord(ctx->ev[2], st);
    ctx->launches += 4;
    std::vector<u8> gok(groups), ok(n);
    CK(cudaMemcpyAsync(gok.data(), d_gok, groups, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(ok.data(), d_ok, n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    // members of failed groups (whose encoding is fine) go through one-by-one verification; their verdicts replace the zeros
    std::vector<u32> idx;
    u32 failed = 0;
    for (u32 g = 0; g < groups; g++) {
        if (gok[g]) continue;
        failed++;
        size_t lo = (size_t)g * SV_SB_GROUP, hi = lo + SV_SB_GROUP < n ? lo + SV_SB_GROUP : n;
        for (size_t i = lo; i < hi; i++)
            if (ok[i]) idx.push_back((u32)i);
    }
    if (groups_total) *groups_total = groups;
    if (groups_failed) *groups_failed = failed;
    if (!idx.empty()) {
        size_t c = idx.size();
        CK(cudaMemcpyAsync(d_idx, idx.data(), 4 * c, cudaMemcpyHostToDevice, st));
        // gathered copies live in the upper halves... of a second staging area: the pts array is dead by now (2n x 96 bytes >= 160 c)
        u8* g_msg = reinterpret_cast<u8*>(d_pts);
        u8* g_key = g_msg + 32 * c;
        u8* g_sig = g_key + 32 * c;
        u8* g_v = g_sig + 64 * c;
        k_sb_gather<<<(unsigned)((c + 255) / 256), 256, 0, st>>>(d_idx, c, ctx->d_msg, ctx->d_key, ctx->d_sig, g_msg, g_key, g_sig);
        ctx->launches += 1;
        rc = launch_verify(ctx, SV_KIND_SCHNORR, g_msg, g_key, g_sig, c, g_v, nullptr, st);
        if (rc) return rc;
        k_mixed_scatter<<<(unsigned)((c + 255) / 256), 256, 0, st>>>(d_idx, c, g_v, d_out);
        ctx->launches += 1;
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(verdicts, d_out, n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SV_OK;
}

// ---- deferral queue -----------------------------------------------------------------------------
extern "C" long sv_enqueue(sv_ctx* ctx, int kind, const uint8_t msg32[32], const uint8_t* key, const uint8_t sig64[64]) {
    size_t ks = sv_key_size(kind);
    if (!ctx || ks == 0 || !msg32 || !key || !sig64) return SV_ERR_ARG;
    sv_queue_item it;
    it.kind = kind;
    memcpy(it.msg, msg32, 32);
    memset(it.key, 0, 64);
    memcpy(it.key, key, ks);
    memcpy(it.sig, sig64, 64);
    ctx->queue.push_back(it);
    return (long)ctx->queue.size() - 1;
}
extern "C" size_t sv_pending(const sv_ctx* ctx) { return ctx ? ctx->queue.size() : 0; }

extern "C" int sv_flush(sv_ctx* ctx, uint8_t* verdicts, size_t capacity) {
    if (!ctx || (!verdicts && !ctx->queue.empty())) return SV_ERR_ARG;
    size_t total = ctx->queue.size();
    if (capacity < total) return SV_ERR_ARG;
    // segregate by kind so that warps stay homogeneous, verify, scatter verdicts back in enqueue order
    for (int kind = 0; kind < 3; kind++) {
        size_t ks = sv_key_size(kind);
        std::vector<size_t> idx;
        for (size_t i = 0; i < total; i++)
            if (ctx->queue[i].kind == kind) idx.push_back(i);
        if (idx.empty()) continue;
        size_t m = idx.size();
        std::vector<u8> msg(32 * m), key(ks * m), sig(64 * m), out(m);
        for (size_t j = 0; j < m; j++) {
            const sv_queue_item& it = ctx->queue[idx[j]];
            memcpy(&msg[32 * j], it.msg, 32);
            memcpy(&key[ks * j], it.key, ks);
            memcpy(&sig[64 * j], it.sig, 64);
        }
        int rc = sv_verify_host(ctx, kind, msg.data(), key.data(), sig.data(), m, out.data());
        if (rc) return rc;
        for (size_t j = 0; j < m; j++) verdicts[idx[j]] = out[j];
    }
    ctx->queue.clear();
    return SV_OK;
}

// ---- self test (test support) ---------------------------------------------------------------------
extern "C" int sv_selftest_host(sv_ctx* ctx, int op, const uint32_t* a, const uint32_t* b, size_t n, uint32_t* out) {
    if (!ctx || op < 0 || op > SV_ST_FE_INV_VAR || (n && (!a || !b || !out))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    dev_tmp ta, tb, to;
    CK(ta.alloc(n * 32));
    CK(tb.alloc(n * 32));
    CK(to.alloc(n * 64));
    cudaStream_t st = ctx->stream;
    CK(cudaMemcpyAsync(ta.p, a, n * 32, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(tb.p, b, n * 32, cudaMemcpyHostToDevice, st));
    k_selftest<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(op, ta.as<u32>(), tb.as<u32>(), n, to.as<u32>(), ctx->d_gtab);
    ctx->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, to.p, n * 64, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SV_OK;
}

// ---- synthetic workload + probes ----------------------------------------------------------------
extern "C" int sv_synth_device(sv_ctx* ctx, int kind, uint64_t seed, size_t n, void* d_msg32, void* d_key,
                               void* d_sig64, void* stream) {
    if (!ctx || sv_key_size(kind) == 0 || (n && (!d_msg32 || !d_key || !d_sig64))) return SV_ERR_ARG;
    if (n == 0) return SV_OK;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    unsigned grid = (unsigned)((n + 127) / 128);
    if (kind == SV_KIND_ECDSA33)
        k_synth<SV_KIND_ECDSA33><<<grid, 128, 0, st>>>(seed, n, ctx->d_gtab, (u8*)d_msg32, (u8*)d_key, (u8*)d_sig64);
    else if (kind == SV_KIND_ECDSA_XY)
        k_synth<SV_KIND_ECDSA_XY><<<grid, 128, 0, st>>>(seed, n, ctx->d_gtab, (u8*)d_msg32, (u8*)d_key, (u8*)d_sig64);
    else
        k_synth<SV_KIND_SCHNORR><<<grid, 128, 0, st>>>(seed, n, ctx->d_gtab, (u8*)d_msg32, (u8*)d_key, (u8*)d_sig64);
    ctx->launches += 1;
    CK(cudaGetLastError());
    return SV_OK;
}

extern "C" int sv_probe(sv_ctx* ctx, int mode, double* ops_per_sec) {
    if (!ctx || !ops_per_sec || mode < 0 || mode > 10) return SV_ERR_ARG;
    dev_guard dg__;
    CK(dg__.enter(ctx->device));
    const int iters = (mode == 2 || mode == 3 || mode >= 9) ? 2000 : 4000;
    // modes 9/10: ONE warp on the whole device — the dependent-chain latency of fe_mul / fe_sqr (small-batch path)
    const int blocks = mode >= 9 ? 1 : ctx->sm_count * 8, threads = mode >= 9 ? 32 : 256;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CK(cudaEventRecord(e0, ctx->stream));
        switch (mode) {
            case 0: k_probe_imad_wide<<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
            case 1: k_probe_cmad4<<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
            case 2: k_probe_fe<0><<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
            case 3: k_probe_fe<1><<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
            case 4: k_probe_chain8<<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
            case 5: k_probe_carry_save<<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
            case 6: k_probe_imad32<<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
            case 8: k_probe_dfma<<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
            case 9: k_probe_fe<0><<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
            case 10: k_probe_fe<1><<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
            default: k_probe_addc<<<blocks, threads, 0, ctx->stream>>>(iters, ctx->d_sink); break;
        }
        CK(cudaEventRecord(e1, ctx->stream));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
        ctx->launches += 1;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    // operations per thread per launch
    static const double per_iter[11] = {32.0, 32.0, 2.0, 2.0, 32.0, 32.0, 32.0, 64.0, 32.0, 2.0, 1.0};  // mode 10: two INDEPENDENT squaring chains -> one chain's rate
    // modes 9/10 report dependent operations per second of ONE thread (the two chains of the probe depend on each other)
    *ops_per_sec = per_iter[mode] * iters * (mode >= 9 ? 1.0 : (double)blocks * threads) / (best * 1e-3);
    return SV_OK;
}
extern "C" int sv_probe_imad_peak(sv_ctx* ctx, double* imad_per_sec) { return sv_probe(ctx, 0, imad_per_sec); }

// pinned host memory for callers that want full-speed H2D/D2H
extern "C" void* sv_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
extern "C" void sv_host_free(void* p) {
    if (p) cudaFreeHost(p);
}
