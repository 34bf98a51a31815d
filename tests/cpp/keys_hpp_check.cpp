// TEST PROGRAM for the key slots of act::Engine and its keyed overload of batch_verify_spend_and_refund (include/act.hpp): reads
// a fixture written by tests/test_key_slots.py, installs the keys it lists, selects one, runs the issuer's loop twice over the same
// slice with ONE shared RNG stream and a store per slot (slots 0 and 3 share one), writes every output byte back.
// usage: keys_hpp_check <fixture.bin> <out.bin>
#include <cstdio>
#include <fstream>
#include <iterator>
#include <memory>

#include "act.hpp"

struct StreamRng {
    const std::vector<uint8_t>& s;
    size_t pos = 0;
    void fill_bytes(uint8_t* dst, size_t n) {
        if (pos + n > s.size()) throw std::runtime_error("rng stream exhausted");
        std::memcpy(dst, s.data() + pos, n);
        pos += n;
    }
};
static uint32_t rd32(const std::vector<uint8_t>& b, size_t& o) { uint32_t v; std::memcpy(&v, b.data() + o, 4); o += 4; return v; }
static void wr(std::vector<uint8_t>& o, const void* p, size_t n) { const uint8_t* q = (const uint8_t*)p; o.insert(o.end(), q, q + n); }
static void wr32(std::vector<uint8_t>& o, uint32_t v) { wr(o, &v, 4); }

int main(int argc, char** argv) {
    if (argc < 3) { std::fprintf(stderr, "usage: %s fixture.bin out.bin\n", argv[0]); return 2; }
    std::ifstream f(argv[1], std::ios::binary);
    std::vector<uint8_t> b((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    size_t o = 0;
    act::Params params;
    std::memcpy(params.h.data(), b.data(), 96); o = 96;
    uint32_t nkeys = rd32(b, o);   // slot, x, w per key; the first is the creation key (slot 0)
    std::vector<std::pair<int, act::PrivateKey>> keys;
    for (uint32_t k = 0; k < nkeys; k++) {
        int slot = (int)rd32(b, o);
        act::Scalar x; act::Bytes32 w;
        std::memcpy(x.data(), b.data() + o, 32); std::memcpy(w.data(), b.data() + o + 32, 32); o += 64;
        keys.emplace_back(slot, act::PrivateKey(x, w));
    }
    int selected = (int)rd32(b, o);
    uint32_t np = rd32(b, o);
    std::vector<act::SpendProof> proofs(np);
    for (uint32_t i = 0; i < np; i++) { std::memcpy(proofs[i].bytes.data(), b.data() + o, ACT_PROOF_BYTES); o += ACT_PROOF_BYTES; }
    std::vector<uint8_t> key_ids(b.begin() + o, b.begin() + o + np); o += np;
    uint32_t nrng = rd32(b, o);
    std::vector<uint8_t> stream(b.begin() + o, b.begin() + o + nrng);

    try {
        act::Engine eng(params, keys[0].second, 0);
        for (size_t k = 1; k < keys.size(); k++) eng.set_key(keys[k].first, keys[k].second);
        eng.select_key(selected);
        std::vector<std::unique_ptr<act::NullifierStore>> owned;
        std::array<act::NullifierStore*, ACT_KEY_SLOTS> stores{};
        for (auto& k : keys) {
            if (k.first == 3 && stores[0]) { stores[3] = stores[0]; continue; }
            owned.emplace_back(new act::NullifierStore(0, 16));
            stores[(size_t)k.first] = owned.back().get();
        }
        StreamRng rng{stream};
        std::vector<uint8_t> out;
        for (int pass = 0; pass < 2; pass++) {                // the second pass replays the whole slice: every accepted proof is Err now
            auto res = eng.batch_verify_spend_and_refund(proofs, key_ids, rng, stores);
            for (auto& r : res) out.push_back(r.status);
            for (auto& r : res) wr(out, r.value.nullifier.data(), 32);
            for (auto& r : res) wr(out, r.value.refund.bytes.data(), ACT_REFUND_BYTES);
            wr32(out, (uint32_t)rng.pos);
        }
        for (auto& s : owned) wr32(out, (uint32_t)s->size());
        std::ofstream g(argv[2], std::ios::binary);
        g.write((const char*)out.data(), (std::streamsize)out.size());
        std::printf("keys_hpp_check ok: %u proofs, %zu rng bytes drawn\n", np, rng.pos);
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "keys_hpp_check FAILED: %s\n", ex.what());
        return 1;
    }
    return 0;
}
