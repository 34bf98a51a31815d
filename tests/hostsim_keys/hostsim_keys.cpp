// hostsim_keys.cpp -- TEST-ONLY: the host build of the device headers (tests/hostsim/hostsim.cpp, included whole) plus the keyed
// spend pipeline of an engine with several issuer keys: the per-thread kernel bodies in plain loops, with the keyed head
// (spend_head_thread<true>) reading each proof's secret from a table of ACT_KEY_SLOTS contexts.  Never linked into libact_b200.so.
#include "../hostsim/hostsim.cpp"

// proof p is verified under the key of slots[key_ids[p]] (ACT_KEY_SLOTS contexts, null = empty slot) and refunded under `sel`
EXPORT void hs_refund_keyed(const hs_ctx* sel, const hs_ctx* const* slots, size_t n, const uint8_t* proofs, const uint8_t* key_ids, const uint8_t* rnd,
                            uint8_t* refunds, uint8_t* nullifiers, uint8_t* status) {
    const act_ctx* c[ACT_KEY_SLOTS];
    for (int k = 0; k < ACT_KEY_SLOTS; k++) c[k] = slots[k] ? &slots[k]->c : nullptr;
    const act_ctx* C = &sel->c;
    auto pf = to_words(proofs, n * (size_t)ACT_PROOF_WORDS * 4), d = to_words(rnd, n * 128);
    std::vector<u32> items(n * (size_t)ACT_ITEM_WORDS + 8), cn(n * (size_t)ACT_L * 24 + 8), kp(n * 32 + 8), flags(n + 1, 0),
        cvs(n * ACT_SPEND_CHUNKS * 8 + 8), ro(n * 32 + 8), no(n * 8 + 8);
    std::vector<vb_table> tabs(ACT_RANGE_SPLIT);
    std::vector<u32> cpts(n * 2 * ACT_L * 32 + 8);
    for (size_t p = 0; p < n; p++)
        for (int j = 0; j < ACT_L; j++) spend_range_thread(C, p, j, pf.data(), items.data(), cn.data(), flags.data(), tabs.data(), cpts.data());
    for (size_t p = 0; p < n; p++) spend_head_thread<true>(C, p, pf.data(), items.data(), cn.data(), kp.data(), flags.data(), cpts.data(), key_ids, c);
    for (size_t p = 0; p < n; p++)
        for (int part = 0; part < 2 * ACT_L / ACT_ENC_BATCH; part++) spend_encode_thread(C, p, part, cpts.data(), items.data());
    for (size_t p = 0; p < n; p++)
        for (int k = 0; k < ACT_SPEND_CHUNKS; k++) spend_chunk_thread(C, p, k, items.data(), cvs.data());
    for (size_t p = 0; p < n; p++) spend_finish_thread(C, p, pf.data(), cvs.data(), flags.data(), status);
    for (size_t p = 0; p < n; p++) refund_sign_thread(C, p, pf.data(), d.data(), kp.data(), status, ro.data(), no.data());
    memcpy(refunds, ro.data(), n * 128);
    memcpy(nullifiers, no.data(), n * 32);
}
