// tests/host_emul/emul_recover.cpp — TEST-ONLY host build of the public-key recovery path (verify.cuh "public-key
// recovery").  It compiles emul.cpp's translation unit (the kernel headers, the pair mailbox that stands in for the warp
// shuffle, the fixed-base table) and adds the two schedules the engine runs recovery on, so that tests/test_recover_emul.py
// can compare them with the reference on a machine without a GPU.  Built into tests/host_emul/libemul_recover.so by
// lightning_b200/build.py; never part of libcln_sigverify.so.
#include "emul.cpp"

extern "C" {

// public-key recovery on the throughput schedule: r inverted in batches of SV_PREP_BATCH (k_prep_recover_inv /
// _finish), Q parked in the work record (k_main<SV_KIND_RECOVER>), keys in batches of SV_FINAL_BATCH (k_final_recover).
// status: 1 / 0 / -1 as int8_t
void emul_recover_batch(const u8* msg, const u8* sig, const u8* recid, size_t n, u8* xy64, int8_t* status) {
    build_gtable_fast();
    std::vector<sv_work> work(n);
    for (size_t base = 0; base < n; base += SV_PREP_BATCH) {
        int cnt = (int)((n - base < SV_PREP_BATCH) ? (n - base) : SV_PREP_BATCH);
        sc r[SV_PREP_BATCH], s[SV_PREP_BATCH], m[SV_PREP_BATCH], rv[SV_PREP_BATCH];
        bool ok[SV_PREP_BATCH], parsed[SV_PREP_BATCH];
        for (int j = 0; j < cnt; j++) {
            recover_parse(r[j], s[j], m[j], ok[j], parsed[j], sig + 64 * (base + j), msg + 32 * (base + j), recid[base + j]);
            rv[j] = r[j];
            if (!ok[j]) { memset(rv[j].v, 0, 32); rv[j].v[0] = 1; }
        }
        sc_batch_inverse(rv, cnt);
        for (int j = 0; j < cnt; j++) recover_finish_prep(work[base + j], ok[j], parsed[j], r[j], s[j], m[j], rv[j]);
    }
    qtab_entry tab[8];
    for (size_t i = 0; i < n; i++) {
        const u32 flags = work[i].flags;
        ge R;
        bool ok = recover_lift(R, sig + 64 * i, recid[i]) && recover_lift_allowed(flags, recid[i]);
        gej Q;
        ecmult_uniform(Q, &work[i], R, g_table.data(), tab);
        recover_park(reinterpret_cast<sv_jac*>(&work[i]), Q, ok, (flags & SV_WF_PARSED) != 0);
    }
    for (size_t base = 0; base < n; base += SV_FINAL_BATCH) {
        int cnt = (int)((n - base < SV_FINAL_BATCH) ? (n - base) : SV_FINAL_BATCH);
        recover_final_batch(xy64 + 64 * base, reinterpret_cast<u8*>(status) + base, reinterpret_cast<const sv_jac*>(work.data()) + base,
                            cnt);
    }
}
// public-key recovery on the small-batch schedule, the half ladders on lane pairs (k_small<SV_KIND_RECOVER, false>)
void emul_recover_small_pair_batch(const u8* msg, const u8* sig, const u8* recid, size_t n, u8* xy64, int8_t* status) {
    build_gtable_fast();
    sv_small_item it;
    for (size_t i = 0; i < n; i++) {
        small_recover_key_side(sig + 64 * i, recid[i], &it);
        small_recover_scalar_side(msg + 32 * i, sig + 64 * i, recid[i], &it);
        for (int half = 0; half < 2; half++) {
            pair_mailbox mb;
            std::thread other([&] { pair_lane L; L.role = 1; L.mb = &mb; small_half_ladder_pair(L, &it, half); });
            pair_lane L;
            L.role = 0;
            L.mb = &mb;
            small_half_ladder_pair(L, &it, half);
            other.join();
        }
        small_comb(&it, g_table.data());
        small_recover_finish(&it, recid[i], xy64 + 64 * i, reinterpret_cast<u8*>(status) + i);
    }
}
}
