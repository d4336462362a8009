// blsgpu.hpp -- C++ host-side mirror of the reference crate's public surface (src/bls.rs) on top of the C ABI (blsgpu.h).
//
// The reference is Rust; no Rust toolchain exists in the build image, so the compiled-language host side above the
// C ABI is this header (the Rust shim a maintainer would add is written out in INTEGRATION.md).  Same names, argument
// meaning and error behaviour as the reference:
//   Parameters / PrivateKey / PublicKey / Signature        src/bls.rs:25-357   (Copy value types holding the crate's own
//                                                          serialisations: 48 B / 96 B ZCash compressed, 32 B LE scalar)
//   PublicKey::aggregate / Signature::aggregate            src/bls.rs:183-195, 288-300   -> std::optional (None on empty)
//   BLS::setup / keygen / sign / verify                    src/bls.rs:391-458            -> Result<T> = value or BLSError
//   hash_to_g2                                             src/bls.rs:477-493
//   BLSError {InvalidSecretKey, InvalidPublicKey, InvalidSignature}   src/bls.rs:359-377
// Header-only; link with -lblsgpu.  All arithmetic runs on the GPU; there is no CPU fallback.
#pragma once
#include <array>
#include <cstdint>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>
#include "blsgpu.h"

namespace blsgpu {

enum class BLSError { InvalidSecretKey, InvalidPublicKey, InvalidSignature };                 // src/bls.rs:359-377
struct SerializationError : std::runtime_error { using std::runtime_error::runtime_error; };  // ark_serialize::SerializationError
struct GpuError : std::runtime_error { using std::runtime_error::runtime_error; };

template <class T> struct Result {                       // Result<T, Box<dyn Error>> of the SignatureScheme trait
    std::optional<T> ok; std::optional<BLSError> err;
    bool is_ok() const { return ok.has_value(); }
    T unwrap() const { if (!ok) throw std::runtime_error("called unwrap() on an Err value"); return *ok; }
    T unwrap_or(T d) const { return ok ? *ok : d; }      // tests/tests.rs:262 collapses Err to false
};

class Context {                                          // one per GPU per process
    blsgpu_ctx* h_ = nullptr;
public:
    explicit Context(int device = -1) { if (blsgpu_create(&h_, device) != 0) throw GpuError("no usable sm_100 CUDA device (libblsgpu has no CPU fallback)"); }
    ~Context() { if (h_) blsgpu_destroy(h_); }
    Context(const Context&) = delete; Context& operator=(const Context&) = delete;
    blsgpu_ctx* raw() const { return h_; }
    void check(int rc) const { if (rc != 0) throw GpuError(blsgpu_last_error(h_)); }
};
inline Context& default_context() { static Context c; return c; }

inline std::vector<uint8_t> from_hex(const std::string& s) {                                  // malformed hex panics in the reference (src/bls.rs:83,230,327)
    size_t o = (s.size() >= 2 && s[0] == '0' && (s[1] == 'x' || s[1] == 'X')) ? 2 : 0;
    if ((s.size() - o) % 2) throw std::invalid_argument("odd-length hex");
    std::vector<uint8_t> out((s.size() - o) / 2);
    auto nib = [](char c) -> int { if (c >= '0' && c <= '9') return c - '0'; c |= 32; if (c >= 'a' && c <= 'f') return c - 'a' + 10; throw std::invalid_argument("bad hex digit"); };
    for (size_t i = 0; i < out.size(); i++) out[i] = (uint8_t)(nib(s[o + 2 * i]) << 4 | nib(s[o + 2 * i + 1]));
    return out;
}
inline std::string to_hex(const uint8_t* p, size_t n) { static const char* d = "0123456789abcdef"; std::string s(2 * n, '0'); for (size_t i = 0; i < n; i++) { s[2 * i] = d[p[i] >> 4]; s[2 * i + 1] = d[p[i] & 15]; } return s; }

struct Parameters { std::array<uint8_t, 48> g1_generator; };                                  // src/bls.rs:26-36

struct PrivateKey {                                                                           // src/bls.rs:53-121, 32-byte little-endian Fr
    std::array<uint8_t, 32> private_key{};
    static PrivateKey try_from(const std::vector<uint8_t>& b) {
        static const uint8_t R_LE[32] = {0x01, 0x00, 0x00, 0x00, 0xff, 0xff, 0xff, 0xff, 0xfe, 0x5b, 0xfe, 0xff, 0x02, 0xa4, 0xbd, 0x53, 0x05, 0xd8, 0xa1, 0x09, 0x08, 0xd8, 0x39, 0x33, 0x48, 0x7d, 0x9d, 0x29, 0x53, 0xa7, 0xed, 0x73};
        if (b.size() < 32) throw SerializationError("short");
        PrivateKey k; std::copy(b.begin(), b.begin() + 32, k.private_key.begin());
        for (int i = 31; i >= 0; i--) { if (k.private_key[i] != R_LE[i]) { if (k.private_key[i] > R_LE[i]) throw SerializationError("not a canonical Fr element"); return k; } }
        throw SerializationError("not a canonical Fr element");
    }
    static PrivateKey try_from(const std::string& hex) { return try_from(from_hex(hex)); }
    std::vector<uint8_t> to_bytes() const { return {private_key.begin(), private_key.end()}; }
    std::string to_hex() const { return blsgpu::to_hex(private_key.data(), 32); }
    bool operator==(const PrivateKey& o) const { return private_key == o.private_key; }
};

struct PublicKey {                                                                            // src/bls.rs:136-260
    std::array<uint8_t, 48> public_key{};
    PublicKey() { public_key[0] = 0xc0; }                                                     // default = identity (src/bls.rs:140-146)
    static PublicKey try_from(const std::vector<uint8_t>& b, Context& c = default_context()) {
        if (b.size() < 48) throw SerializationError("short");
        uint8_t code = 0; c.check(blsgpu_deserialize_g1(c.raw(), b.data(), 1, &code));        // reads exactly 48 bytes like ark-serialize
        if (code > BLSGPU_DE_INFINITY) throw SerializationError("invalid G1 encoding");
        PublicKey k; if (code == BLSGPU_DE_OK) std::copy(b.begin(), b.begin() + 48, k.public_key.begin());
        return k;
    }
    static PublicKey try_from(const std::string& hex, Context& c = default_context()) { return try_from(from_hex(hex), c); }
    static PublicKey from(const PrivateKey& sk, Context& c = default_context()) {            // From<&PrivateKey>, src/bls.rs:210-216
        PublicKey k; c.check(blsgpu_sk_to_pk_batch(c.raw(), sk.private_key.data(), 1, k.public_key.data(), nullptr)); return k;
    }
    static std::optional<PublicKey> aggregate(const std::vector<PublicKey>& keys, Context& c = default_context()) {   // src/bls.rs:183-195
        if (keys.empty()) return std::nullopt;
        std::vector<uint8_t> buf(48 * keys.size()); for (size_t i = 0; i < keys.size(); i++) std::copy(keys[i].public_key.begin(), keys[i].public_key.end(), buf.begin() + 48 * i);
        uint32_t seg[2] = {0, (uint32_t)keys.size()}; uint8_t st = 0; PublicKey out;
        c.check(blsgpu_g1_aggregate(c.raw(), buf.data(), seg, 1, out.public_key.data(), &st));
        if (st != 0) throw SerializationError("aggregate member failed to decode");
        return out;
    }
    std::vector<uint8_t> to_bytes() const { return {public_key.begin(), public_key.end()}; }
    std::string to_hex() const { return blsgpu::to_hex(public_key.data(), 48); }
    bool operator==(const PublicKey& o) const { return public_key == o.public_key; }
};

struct Signature {                                                                            // src/bls.rs:263-357
    std::array<uint8_t, 96> sig{};
    Signature() { sig[0] = 0xc0; }
    static Signature try_from(const std::vector<uint8_t>& b, Context& c = default_context()) {
        if (b.size() < 96) throw SerializationError("short");
        uint8_t code = 0; c.check(blsgpu_deserialize_g2(c.raw(), b.data(), 1, &code));
        if (code > BLSGPU_DE_INFINITY) throw SerializationError("invalid G2 encoding");
        Signature s; if (code == BLSGPU_DE_OK) std::copy(b.begin(), b.begin() + 96, s.sig.begin());
        return s;
    }
    static Signature try_from(const std::string& hex, Context& c = default_context()) { return try_from(from_hex(hex), c); }
    static std::optional<Signature> aggregate(const std::vector<Signature>& sigs, Context& c = default_context()) {   // src/bls.rs:288-300
        if (sigs.empty()) return std::nullopt;
        std::vector<uint8_t> buf(96 * sigs.size()); for (size_t i = 0; i < sigs.size(); i++) std::copy(sigs[i].sig.begin(), sigs[i].sig.end(), buf.begin() + 96 * i);
        uint32_t seg[2] = {0, (uint32_t)sigs.size()}; uint8_t st = 0; Signature out;
        c.check(blsgpu_g2_aggregate(c.raw(), buf.data(), seg, 1, out.sig.data(), &st));
        if (st != 0) throw SerializationError("aggregate member failed to decode");
        return out;
    }
    std::vector<uint8_t> to_bytes() const { return {sig.begin(), sig.end()}; }
    std::string to_hex() const { return blsgpu::to_hex(sig.data(), 96); }
    bool operator==(const Signature& o) const { return sig == o.sig; }
};

inline Signature hash_to_g2(const uint8_t* msg, size_t len, Context& c = default_context()) { // src/bls.rs:477-493
    uint32_t off[2] = {0, (uint32_t)len}; Signature s; uint8_t dummy = 0;
    c.check(blsgpu_hash_to_g2_batch(c.raw(), len ? msg : &dummy, off, 1, s.sig.data())); return s;
}

struct BLS {                                                                                  // impl SignatureScheme for BLS<P>, src/bls.rs:379-475
    static Parameters setup() {                                                               // src/bls.rs:391-393
        Parameters p; auto g = from_hex("97f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb");
        std::copy(g.begin(), g.end(), p.g1_generator.begin()); return p;
    }
    template <class Rng> static Result<std::pair<PublicKey, PrivateKey>> keygen(const Parameters&, Rng& rng, Context& c = default_context()) {   // src/bls.rs:395-409
        PrivateKey sk; for (auto& b : sk.private_key) b = (uint8_t)rng(); sk.private_key[31] &= 0x3f;          // a canonical Fr element
        return {std::make_pair(PublicKey::from(sk, c), sk), std::nullopt};
    }
    static Result<Signature> sign(const Parameters&, const PrivateKey& sk, const uint8_t* msg, size_t len, Context& c = default_context()) {   // src/bls.rs:411-425
        uint32_t off[2] = {0, (uint32_t)len}; Signature s; uint8_t st = 0, dummy = 0;
        c.check(blsgpu_sign_batch(c.raw(), sk.private_key.data(), len ? msg : &dummy, off, 1, s.sig.data(), &st));
        if (st == BLSGPU_ST_BAD_SECKEY) return {std::nullopt, BLSError::InvalidSecretKey};
        return {s, std::nullopt};
    }
    static Result<bool> verify(const Parameters&, const PublicKey& pk, const uint8_t* msg, size_t len, const Signature& sig, Context& c = default_context()) {   // src/bls.rs:427-458
        uint32_t off[2] = {0, (uint32_t)len}; uint8_t st = 0, dummy = 0;
        c.check(blsgpu_verify_batch(c.raw(), pk.public_key.data(), len ? msg : &dummy, off, sig.sig.data(), 1, &st, nullptr, nullptr));
        if (st == BLSGPU_ST_BAD_PUBKEY) return {std::nullopt, BLSError::InvalidPublicKey};
        if (st == BLSGPU_ST_BAD_SIG) return {std::nullopt, BLSError::InvalidSignature};
        return {st == BLSGPU_ST_TRUE, std::nullopt};
    }
    // batch-first form (no reference counterpart): status per item, ok-bitmap, optional GT accumulator
    static std::vector<uint8_t> verify_batch(const std::vector<uint8_t>& pk48, const std::vector<uint8_t>& msg32, const std::vector<uint8_t>& sig96, Context& c = default_context()) {
        size_t n = sig96.size() / 96; std::vector<uint8_t> st(n);
        c.check(blsgpu_verify_batch(c.raw(), pk48.data(), msg32.data(), nullptr, sig96.data(), n, st.data(), nullptr, nullptr)); return st;
    }
    // signature sets (no reference counterpart; blsgpu_verify_signature_sets): set s = keys [key_off[s], key_off[s+1]) of pks48, message
    // msg[msg_off[s] .. msg_off[s+1]), signature s -> status per set.  seed16 (nullable): random-linear-combination form with the exact outcome.
    static std::vector<uint8_t> verify_signature_sets(const std::vector<uint8_t>& pks48, const std::vector<uint32_t>& key_off, const std::vector<uint8_t>& msg,
                                                      const std::vector<uint32_t>& msg_off, const std::vector<uint8_t>& sig96, const uint8_t* seed16 = nullptr,
                                                      const uint64_t* bitmap = nullptr, uint64_t* fallback_sets = nullptr, Context& c = default_context()) {
        size_t n = sig96.size() / 96; std::vector<uint8_t> st(n);
        if (key_off.size() != n + 1 || msg_off.size() != n + 1 || key_off[n] > pks48.size() / 48 || msg_off[n] > msg.size()) throw std::invalid_argument("key_off / msg_off do not match the buffers");
        uint8_t dummy = 0;
        c.check(blsgpu_verify_signature_sets(c.raw(), pks48.empty() ? &dummy : pks48.data(), key_off.data(), bitmap, msg.empty() ? &dummy : msg.data(), msg_off.data(),
                                             sig96.data(), n, seed16, st.data(), nullptr, fallback_sets));
        return st;
    }
};

}  // namespace blsgpu
