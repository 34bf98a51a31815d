// TEST PROGRAM for act::NullifierStore and the store overload of act::Engine::batch_verify_spend_and_refund (include/act.hpp):
// reads a fixture written by tests/test_nullifier_store.py, imports a prefill set into a store, runs the issuer's loop twice over
// the same slice with ONE shared RNG stream, writes every output byte back.
// usage: store_hpp_check <fixture.bin> <out.bin> [device0,device1]
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iterator>
#include <sstream>

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
    if (argc < 3) { std::fprintf(stderr, "usage: %s fixture.bin out.bin [devices]\n", argv[0]); return 2; }
    std::ifstream f(argv[1], std::ios::binary);
    std::vector<uint8_t> b((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    size_t o = 0;
    act::Params params;
    std::memcpy(params.h.data(), b.data(), 96); o = 96;
    act::Scalar x; act::Bytes32 w;
    std::memcpy(x.data(), b.data() + o, 32); std::memcpy(w.data(), b.data() + o + 32, 32); o += 64;
    uint32_t np = rd32(b, o);
    std::vector<act::SpendProof> proofs(np);
    for (uint32_t i = 0; i < np; i++) { std::memcpy(proofs[i].bytes.data(), b.data() + o, ACT_PROOF_BYTES); o += ACT_PROOF_BYTES; }
    uint32_t nseen = rd32(b, o);
    std::vector<uint8_t> seen(b.begin() + o, b.begin() + o + 32 * (size_t)nseen); o += 32 * (size_t)nseen;
    uint32_t nrng = rd32(b, o);
    std::vector<uint8_t> stream(b.begin() + o, b.begin() + o + nrng);

    try {
        act::PrivateKey key(x, w);
        std::vector<int> devices;
        if (argc > 3) { std::stringstream ss(argv[3]); std::string t; while (std::getline(ss, t, ',')) devices.push_back(std::atoi(t.c_str())); }
        act::Engine eng = devices.empty() ? act::Engine(params, key, 0) : act::Engine(params, key, devices);
        act::NullifierStore store(devices.empty() ? 0 : devices[0], 16);
        std::vector<uint8_t> st0(nseen, 0);
        store.screen(st0, seen, true);                        // bulk import of the keys spent before this slice
        StreamRng rng{stream};
        std::vector<uint8_t> out;
        for (int pass = 0; pass < 2; pass++) {                // the second pass replays the whole slice: every proof is Err now
            auto res = eng.batch_verify_spend_and_refund(proofs, rng, store);
            for (auto& r : res) out.push_back(r.status);
            for (auto& r : res) wr(out, r.value.nullifier.data(), 32);
            for (auto& r : res) wr(out, r.value.refund.bytes.data(), ACT_REFUND_BYTES);
            wr32(out, (uint32_t)rng.pos);
        }
        wr32(out, (uint32_t)store.size());
        auto members = store.members();
        wr32(out, (uint32_t)members.size());
        for (auto& m : members) wr(out, m.data(), 32);
        std::ofstream g(argv[2], std::ios::binary);
        g.write((const char*)out.data(), (std::streamsize)out.size());
        std::printf("store_hpp_check ok: %u proofs, %zu members, %zu rng bytes drawn\n", np, members.size(), rng.pos);
    } catch (const std::exception& ex) {
        std::fprintf(stderr, "store_hpp_check FAILED: %s\n", ex.what());
        return 1;
    }
    return 0;
}
