// act.hpp -- C++ host-side mirror of the reference crate's interface for the hot path, over the C ABI of act_engine.h.
//
// The reference (/root/reference, Rust) exposes the path as methods on its own types:
//     Params::new(org, service, deployment, version)                                   src/lib.rs:291-315
//     PrivateKey::issue(&params, &request, c, rng)  -> Result<IssuanceResponse, Error>  src/lib.rs:621-663
//     PrivateKey::refund(&params, &spend_proof, rng) -> Result<Refund, Error>           src/lib.rs:781-869
//     SpendProof::nullifier()                                                           src/lib.rs:720-722
//     PreIssuance::to_credit_token / PreRefund::to_credit_token (verification halves)   src/lib.rs:528-562, 1217-1253
//     to_cbor / from_cbor on every wire type                                            src/cbor.rs:94-465
// A Rust `-sys` + wrapper crate is the intended host (rust/, INTEGRATION.md) but cannot be compiled in this image; this header is
// the same wrapper in C++: same names, same argument meaning, the same per-request `Result<T, Error>` (act::Result), the same RNG
// behaviour (e and alpha -- 64 bytes each -- are drawn only for requests that verified, in slice order: src/lib.rs:638-643, 842-846),
// as `batch_issue` / `batch_verify_spend_and_refund` over slices.  Header-only; link with libact_b200.so.  No CPU fallback.
#ifndef ACT_HPP
#define ACT_HPP

#include <array>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "act_engine.h"

namespace act {

using Bytes32 = std::array<uint8_t, 32>;
using Scalar = Bytes32;   // 32-byte little-endian scalar as on the wire (reduced mod l by the engine: src/cbor.rs:80-91)

// `Error` of the reference, same order and meaning (src/lib.rs:102-112); status byte = 1 + discriminant
enum class Error : uint8_t {
    InvalidIssuanceRequestProof = 1, InvalidIssuanceResponseProof = 2, DoubleSpendError = 3, InvalidRefundProof = 4,
    InvalidRefundResponseProof = 5, IdentityPointError = 6, InvalidClientSpendProof = 7, AmountTooBigError = 8, ScalarOutOfRangeError = 9,
    // CborError of src/cbor.rs:30-37 as the engine reports it
    CborInvalidPoint = 0x81, CborInvalidStructure = 0x82, CborParse = 0x83,
};
inline const char* to_string(Error e) {
    switch (e) {
        case Error::InvalidIssuanceRequestProof: return "InvalidIssuanceRequestProof";
        case Error::InvalidIssuanceResponseProof: return "InvalidIssuanceResponseProof";
        case Error::DoubleSpendError: return "DoubleSpendError";
        case Error::InvalidRefundProof: return "InvalidRefundProof";
        case Error::InvalidRefundResponseProof: return "InvalidRefundResponseProof";
        case Error::IdentityPointError: return "IdentityPointError";
        case Error::InvalidClientSpendProof: return "InvalidClientSpendProof";
        case Error::AmountTooBigError: return "AmountTooBigError";
        case Error::ScalarOutOfRangeError: return "ScalarOutOfRangeError";
        case Error::CborInvalidPoint: return "CborError::InvalidValue(invalid Ristretto point)";
        case Error::CborInvalidStructure: return "CborError::InvalidStructure";
        case Error::CborParse: return "CborError::Ciborium";
    }
    return "?";
}

// Result<T, Error>: `ok()` <=> status byte 0; `value` is zero-filled otherwise
template <typename T>
struct Result {
    uint8_t status = 0;
    T value{};
    bool ok() const { return status == 0; }
    Error error() const { return static_cast<Error>(status); }
    const T& unwrap() const {
        if (!ok()) throw std::runtime_error(std::string("act::Result::unwrap on Err(") + to_string(error()) + ")");
        return value;
    }
};

struct EngineError : std::runtime_error {
    explicit EngineError(const std::string& what) : std::runtime_error(what + ": " + act_last_error()) {}
};

// ---- wire types (fixed records of act_engine.h; CBOR forms of src/cbor.rs) ----------------------------------------------
struct IssuanceRequest {   // K | gamma | k_bar | r_bar                      src/lib.rs:376-385
    std::array<uint8_t, ACT_REQUEST_BYTES> bytes{};
    std::vector<uint8_t> to_cbor() const { std::vector<uint8_t> o(ACT_CBOR_REQUEST_BYTES); o.resize(act_encode_issuance_request_cbor(bytes.data(), o.data())); return o; }
    static Result<IssuanceRequest> from_cbor(const uint8_t* p, size_t n) {
        Result<IssuanceRequest> r;
        act_pack_issuance_requests_cbor(1, &p, &n, r.value.bytes.data(), &r.status);
        return r;
    }
};
struct IssuanceResponse {  // A | e | gamma | z | c                           src/lib.rs:572-583
    std::array<uint8_t, ACT_RESPONSE_BYTES> bytes{};
    std::vector<uint8_t> to_cbor() const { std::vector<uint8_t> o(ACT_CBOR_RESPONSE_BYTES); o.resize(act_encode_issuance_response_cbor(bytes.data(), o.data())); return o; }
    static Result<IssuanceResponse> from_cbor(const uint8_t* p, size_t n) {
        Result<IssuanceResponse> r;
        act_pack_issuance_responses_cbor(1, &p, &n, r.value.bytes.data(), &r.status);
        return r;
    }
};
struct SpendProof {        // 526 x 32 bytes in the field order of src/lib.rs:673-708
    std::array<uint8_t, ACT_PROOF_BYTES> bytes{};
    Scalar nullifier_bytes() const { Scalar k; std::memcpy(k.data(), bytes.data(), 32); return k; }   // as sent; the engine returns the reduced value
    Scalar charge() const { Scalar s; std::memcpy(s.data(), bytes.data() + 32, 32); return s; }         // src/lib.rs:729-731
    const uint8_t* com() const { return bytes.data() + 4 * 32; }                                       // com[128], 4096 bytes
    std::vector<uint8_t> to_cbor() const { std::vector<uint8_t> o(ACT_CBOR_PROOF_BYTES); o.resize(act_encode_spend_proof_cbor(bytes.data(), o.data())); return o; }
    static Result<SpendProof> from_cbor(const uint8_t* p, size_t n) {
        Result<SpendProof> r;
        act_pack_spend_proofs_cbor(1, &p, &n, r.value.bytes.data(), &r.status);
        return r;
    }
};
struct Refund {            // A* | e* | gamma | z                             src/lib.rs:1161-1170
    std::array<uint8_t, ACT_REFUND_BYTES> bytes{};
    std::vector<uint8_t> to_cbor() const { std::vector<uint8_t> o(ACT_CBOR_REFUND_BYTES); o.resize(act_encode_refund_cbor(bytes.data(), o.data())); return o; }
    static Result<Refund> from_cbor(const uint8_t* p, size_t n) {
        Result<Refund> r;
        act_pack_refunds_cbor(1, &p, &n, r.value.bytes.data(), &r.status);
        return r;
    }
};
struct RefundWithNullifier {
    Scalar nullifier{};     // SpendProof::nullifier(), reduced mod l
    Refund refund;
};

// ---- Params, keys -------------------------------------------------------------------------------------------------------
struct Params {            // H1 | H2 | H3 encodings                          src/lib.rs:222-229
    std::array<uint8_t, 96> h{};
    static Params create(const std::string& organization, const std::string& service, const std::string& deployment_id, const std::string& version,
                         int device = 0) {   // Params::new
        Params p;
        if (act_params_derive(device, organization.c_str(), service.c_str(), deployment_id.c_str(), version.c_str(), p.h.data())) throw EngineError("act_params_derive");
        return p;
    }
};
struct PublicKey {
    Bytes32 w{};
};
class PrivateKey {         // x and W = G*x; zeroised on destruction like the reference's (ZeroizeOnDrop, src/lib.rs:160)
  public:
    PrivateKey(const Scalar& x, const Bytes32& w) : x_(x) { pub_.w = w; }
    static PrivateKey from_secret(const Scalar& x, int device = 0) {
        Bytes32 w;
        if (act_public_key(device, x.data(), w.data())) throw EngineError("act_public_key");
        return PrivateKey(x, w);
    }
    PrivateKey(const PrivateKey&) = default;
    ~PrivateKey() { volatile uint8_t* p = x_.data(); for (size_t i = 0; i < x_.size(); i++) p[i] = 0; }
    const PublicKey& public_key() const { return pub_; }    // PrivateKey::public, src/lib.rs:201
    const Scalar& secret() const { return x_; }
  private:
    Scalar x_;
    PublicKey pub_;
};

// ---- the spent set: the caller's NullifierDb (examples/act.rs:60-77), resident on one GPU ---------------------------------------
class NullifierStore {
  public:
    explicit NullifierStore(int device = 0, size_t capacity = size_t(1) << 20) {
        if (act_nullifier_store_create(&s_, device, capacity)) throw EngineError("act_nullifier_store_create");
    }
    NullifierStore(const NullifierStore&) = delete;
    NullifierStore& operator=(const NullifierStore&) = delete;
    ~NullifierStore() { act_nullifier_store_destroy(s_); }
    act_nullifier_store* raw() { return s_; }
    int device() const { return act_nullifier_store_device(s_); }
    size_t size() const { return act_nullifier_store_size(s_); }
    // status-0 entries whose nullifier is in the store or earlier in the slice become 3 (DoubleSpendError); record: insert the
    // nullifiers that keep 0.  `status` is updated in place.
    void screen(std::vector<uint8_t>& status, const std::vector<uint8_t>& nullifiers, bool record = true) {
        size_t n = status.size();
        if (nullifiers.size() != n * 32) throw std::invalid_argument("NullifierStore::screen: 32 bytes of nullifier per status");
        if (act_nullifier_store_screen(s_, n, status.data(), nullifiers.data(), status.data(), record ? 1 : 0)) throw EngineError("act_nullifier_store_screen");
    }
    std::vector<Bytes32> members() {
        size_t cap = size(), count = 0;
        std::vector<Bytes32> out(cap);
        if (act_nullifier_store_export(s_, cap ? out[0].data() : nullptr, cap, &count)) throw EngineError("act_nullifier_store_export");
        out.resize(count);
        return out;
    }
  private:
    act_nullifier_store* s_ = nullptr;
};

// ---- the engine: batch forms of the issuer-side calls ------------------------------------------------------------------------
// Rng: anything with `void fill_bytes(uint8_t* dst, size_t n)` (the reference's `impl CryptoRngCore`).
class Engine {
  public:
    Engine(const Params& params, const PrivateKey& key, int device = 0) {
        if (act_engine_create(&e_, device, params.h.data(), key.secret().data(), key.public_key().w.data())) throw EngineError("act_engine_create");
    }
    // one handle over several GPUs of the box: every call below shards the slice contiguously over one replica per device
    Engine(const Params& params, const PrivateKey& key, const std::vector<int>& devices) {
        if (act_engine_create_multi(&e_, devices.data(), (int)devices.size(), params.h.data(), key.secret().data(), key.public_key().w.data()))
            throw EngineError("act_engine_create_multi");
    }
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;
    ~Engine() { act_engine_destroy(e_); }
    act_engine* raw() { return e_; }

    // n x PrivateKey::issue over ONE rng: outputs, and the rng's state afterwards, equal a loop of reference calls
    template <typename Rng>
    std::vector<Result<IssuanceResponse>> batch_issue(const std::vector<IssuanceRequest>& reqs, const std::vector<Scalar>& cs, Rng& rng) {
        size_t n = reqs.size();
        if (cs.size() != n) throw std::invalid_argument("batch_issue: one credit amount per request");
        std::vector<uint8_t> status(n), resp(n * ACT_RESPONSE_BYTES);
        const uint8_t* rq = n ? reqs[0].bytes.data() : nullptr;      // std::array members are contiguous: the vector IS the n x 128 record array
        const uint8_t* c = n ? cs[0].data() : nullptr;
        if (act_batch_issue_verify(e_, n, rq, status.data())) throw EngineError("act_batch_issue_verify");
        std::vector<uint8_t> rnd = draw(status, rng);
        if (act_batch_issue_sign(e_, n, rq, c, status.data(), rnd.data(), rnd.size(), resp.data())) throw EngineError("act_batch_issue_sign");
        wipe(rnd);
        std::vector<Result<IssuanceResponse>> out(n);
        for (size_t i = 0; i < n; i++) { out[i].status = status[i]; std::memcpy(out[i].value.bytes.data(), resp.data() + i * ACT_RESPONSE_BYTES, ACT_RESPONSE_BYTES); }
        return out;
    }
    // n x (spend-proof verification + PrivateKey::refund), with SpendProof::nullifier() of every accepted proof
    template <typename Rng>
    std::vector<Result<RefundWithNullifier>> batch_verify_spend_and_refund(const std::vector<SpendProof>& proofs, Rng& rng) {
        size_t n = proofs.size();
        std::vector<uint8_t> status(n), nul(n * 32), kprime(n * 128), refunds(n * ACT_REFUND_BYTES);
        const uint8_t* pf = n ? proofs[0].bytes.data() : nullptr;
        if (act_batch_spend_verify(e_, n, pf, nul.data(), status.data(), kprime.data())) throw EngineError("act_batch_spend_verify");
        std::vector<uint8_t> rnd = draw(status, rng);
        if (act_batch_refund_sign(e_, n, kprime.data(), status.data(), rnd.data(), rnd.size(), refunds.data())) throw EngineError("act_batch_refund_sign");
        wipe(rnd);
        std::vector<Result<RefundWithNullifier>> out(n);
        for (size_t i = 0; i < n; i++) {
            out[i].status = status[i];
            std::memcpy(out[i].value.nullifier.data(), nul.data() + 32 * i, 32);
            std::memcpy(out[i].value.refund.bytes.data(), refunds.data() + i * ACT_REFUND_BYTES, ACT_REFUND_BYTES);
        }
        return out;
    }
    // the issuer's loop of examples/act.rs:60-77 over ONE rng with the spent set in `store`: verify, check the nullifier (a replay of
    // the store or of the slice is Err(DoubleSpendError) and gets no refund), refund -- 128 bytes drawn only for the survivors, in
    // slice order -- and record.  Outputs, the rng's state and the store afterwards equal that loop's.
    template <typename Rng>
    std::vector<Result<RefundWithNullifier>> batch_verify_spend_and_refund(const std::vector<SpendProof>& proofs, Rng& rng, NullifierStore& store) {
        size_t n = proofs.size();
        std::vector<uint8_t> status(n), nul(n * 32), kprime(n * 128), refunds(n * ACT_REFUND_BYTES);
        const uint8_t* pf = n ? proofs[0].bytes.data() : nullptr;
        if (act_batch_spend_verify(e_, n, pf, nul.data(), status.data(), kprime.data())) throw EngineError("act_batch_spend_verify");
        store.screen(status, nul, true);
        std::vector<uint8_t> rnd = draw(status, rng);
        if (act_batch_refund_sign(e_, n, kprime.data(), status.data(), rnd.data(), rnd.size(), refunds.data())) throw EngineError("act_batch_refund_sign");
        wipe(rnd);
        std::vector<Result<RefundWithNullifier>> out(n);
        for (size_t i = 0; i < n; i++) {
            out[i].status = status[i];
            std::memcpy(out[i].value.nullifier.data(), nul.data() + 32 * i, 32);
            std::memcpy(out[i].value.refund.bytes.data(), refunds.data() + i * ACT_REFUND_BYTES, ACT_REFUND_BYTES);
        }
        return out;
    }
    // key rotation (include/act_engine.h, issuer key slots): install, select and retire keys; the selected key issues and refunds
    void set_key(int slot, const PrivateKey& key) {
        if (act_engine_set_key(e_, slot, key.secret().data(), key.public_key().w.data())) throw EngineError("act_engine_set_key");
    }
    void clear_key(int slot) { if (act_engine_clear_key(e_, slot)) throw EngineError("act_engine_clear_key"); }
    void select_key(int slot) { if (act_engine_select_key(e_, slot)) throw EngineError("act_engine_select_key"); }
    int selected_key() const { return act_engine_selected_key(e_); }
    uint32_t key_slots() const { return act_engine_key_slots(e_); }
    // the loop above for an issuer with several keys, over ONE rng: proof i is verified under the key of slot key_ids[i], its nullifier
    // is checked against stores[key_ids[i]] (a replay of that store or of an earlier proof of the same store is Err(DoubleSpendError)),
    // and the survivors -- 128 bytes drawn for each, in slice order -- are refunded under the selected key and recorded.  Every slot
    // that holds a key needs a store; slots may share one.  Every store is screened once without recording before any records,
    // so a failure leaves the stores as they were.
    template <typename Rng>
    std::vector<Result<RefundWithNullifier>> batch_verify_spend_and_refund(const std::vector<SpendProof>& proofs, const std::vector<uint8_t>& key_ids,
                                                                           Rng& rng, const std::array<NullifierStore*, ACT_KEY_SLOTS>& stores) {
        size_t n = proofs.size();
        if (key_ids.size() != n) throw std::invalid_argument("keyed call: one key id per proof");
        uint32_t held = key_slots();
        std::vector<NullifierStore*> distinct;
        std::array<int, ACT_KEY_SLOTS> of_slot;
        of_slot.fill(-1);
        for (int k = 0; k < ACT_KEY_SLOTS; k++) {
            if (!(held >> k & 1u)) continue;
            if (!stores[k]) throw std::invalid_argument("keyed call: every slot that holds a key needs a store");
            size_t j = 0;
            while (j < distinct.size() && distinct[j] != stores[k]) j++;
            if (j == distinct.size()) distinct.push_back(stores[k]);
            of_slot[k] = (int)j;
        }
        std::vector<uint8_t> status(n), nul(n * 32), kprime(n * 128), refunds(n * ACT_REFUND_BYTES);
        const uint8_t* pf = n ? proofs[0].bytes.data() : nullptr;
        if (act_batch_spend_verify_keyed(e_, n, pf, key_ids.data(), nul.data(), status.data(), kprime.data())) throw EngineError("act_batch_spend_verify_keyed");
        // each store sees the statuses of its own proofs; the others are nonzero and take no part
        auto store_of = [&](size_t i) { return key_ids[i] < ACT_KEY_SLOTS ? of_slot[key_ids[i]] : -1; };
        std::vector<std::vector<uint8_t>> mine(distinct.size(), std::vector<uint8_t>(n, 0xFF));
        for (size_t i = 0; i < n; i++) if (store_of(i) >= 0) mine[(size_t)store_of(i)][i] = status[i];
        for (size_t j = 0; j < distinct.size(); j++) { std::vector<uint8_t> dry = mine[j]; distinct[j]->screen(dry, nul, false); }
        for (size_t j = 0; j < distinct.size(); j++) distinct[j]->screen(mine[j], nul, true);
        for (size_t i = 0; i < n; i++) if (store_of(i) >= 0) status[i] = mine[(size_t)store_of(i)][i];
        std::vector<uint8_t> rnd = draw(status, rng);
        if (act_batch_refund_sign(e_, n, kprime.data(), status.data(), rnd.data(), rnd.size(), refunds.data())) throw EngineError("act_batch_refund_sign");
        wipe(rnd);
        std::vector<Result<RefundWithNullifier>> out(n);
        for (size_t i = 0; i < n; i++) {
            out[i].status = status[i];
            std::memcpy(out[i].value.nullifier.data(), nul.data() + 32 * i, 32);
            std::memcpy(out[i].value.refund.bytes.data(), refunds.data() + i * ACT_REFUND_BYTES, ACT_REFUND_BYTES);
        }
        return out;
    }
    // the same behind the caller's nullifier check (examples/act.rs:60-77): a proof whose nullifier occurred earlier in the slice or
    // in `seen` is Err(DoubleSpendError) and gets no refund.  Randomness is per request here (rnd: n x 128 bytes).
    std::vector<Result<RefundWithNullifier>> batch_verify_spend_and_refund_screened(const std::vector<SpendProof>& proofs, const std::vector<uint8_t>& rnd,
                                                                                      const std::vector<Scalar>& seen) {
        size_t n = proofs.size();
        if (rnd.size() != n * ACT_RND_BYTES) throw std::invalid_argument("screened call: 128 bytes of randomness per proof");
        std::vector<uint8_t> status(n), nul(n * 32), refunds(n * ACT_REFUND_BYTES);
        if (act_batch_verify_spend_and_refund_screened(e_, n, n ? proofs[0].bytes.data() : nullptr, rnd.data(), seen.size(), seen.empty() ? nullptr : seen[0].data(),
                                                       refunds.data(), nul.data(), status.data()))
            throw EngineError("act_batch_verify_spend_and_refund_screened");
        std::vector<Result<RefundWithNullifier>> out(n);
        for (size_t i = 0; i < n; i++) {
            out[i].status = status[i];
            std::memcpy(out[i].value.nullifier.data(), nul.data() + 32 * i, 32);
            std::memcpy(out[i].value.refund.bytes.data(), refunds.data() + i * ACT_REFUND_BYTES, ACT_REFUND_BYTES);
        }
        return out;
    }
    // verification halves of PreIssuance::to_credit_token / PreRefund::to_credit_token: Ok or the reference's error
    std::vector<uint8_t> batch_issuance_check(const std::vector<IssuanceRequest>& reqs, const std::vector<IssuanceResponse>& resps) {
        size_t n = reqs.size();
        if (resps.size() != n) throw std::invalid_argument("batch_issuance_check: one response per request");
        std::vector<uint8_t> K(n * 32), st(n);
        for (size_t i = 0; i < n; i++) std::memcpy(K.data() + 32 * i, reqs[i].bytes.data(), 32);
        if (act_batch_issuance_check(e_, n, K.data(), n ? resps[0].bytes.data() : nullptr, st.data())) throw EngineError("act_batch_issuance_check");
        return st;
    }
    std::vector<uint8_t> batch_refund_check(const std::vector<SpendProof>& proofs, const std::vector<Refund>& refunds) {
        size_t n = proofs.size();
        if (refunds.size() != n) throw std::invalid_argument("batch_refund_check: one refund per proof");
        std::vector<uint8_t> com(n * ACT_COM_BYTES), st(n);
        for (size_t i = 0; i < n; i++) std::memcpy(com.data() + ACT_COM_BYTES * i, proofs[i].com(), ACT_COM_BYTES);
        if (act_batch_refund_check(e_, n, com.data(), n ? refunds[0].bytes.data() : nullptr, st.data())) throw EngineError("act_batch_refund_check");
        return st;
    }

  private:
    // 128 bytes per ACCEPTED request, in slice order, one 64-byte draw per Scalar::random (e, then alpha) as the reference does
    template <typename Rng>
    static std::vector<uint8_t> draw(const std::vector<uint8_t>& status, Rng& rng) {
        size_t accepted = 0;
        for (uint8_t s : status) accepted += s == 0;
        std::vector<uint8_t> rnd(accepted * ACT_RND_BYTES);
        for (size_t off = 0; off < rnd.size(); off += 64) rng.fill_bytes(rnd.data() + off, 64);
        return rnd;
    }
    static void wipe(std::vector<uint8_t>& v) { volatile uint8_t* p = v.data(); for (size_t i = 0; i < v.size(); i++) p[i] = 0; }
    act_engine* e_ = nullptr;
};

static_assert(sizeof(IssuanceRequest) == ACT_REQUEST_BYTES && sizeof(IssuanceResponse) == ACT_RESPONSE_BYTES && sizeof(SpendProof) == ACT_PROOF_BYTES &&
              sizeof(Refund) == ACT_REFUND_BYTES && sizeof(Scalar) == 32, "wire types are the fixed records of act_engine.h, contiguous in a vector");

}  // namespace act
#endif  // ACT_HPP
