// C++ host-side mirror of the reference's verify-path API over the C ABI (include/jjschnorr_b200.h).
// Same type names, argument meaning and error behaviour as dusk-network/jubjub-schnorr:
//   PublicKey::from_bytes / to_bytes / verify            reference src/keys/public.rs:80-135
//   PublicKeyDouble / SignatureDouble                    reference src/keys/public/double.rs, src/signatures/double.rs
//   PublicKeyVarGen / SignatureVarGen                    reference src/keys/public/var_gen.rs, src/signatures/var_gen.rs
//   multisig::aggregate_pk                               reference src/multisig.rs:154-156
//   Error                                                reference src/error.rs:13-26
//   verify_batch(&[(PublicKey, Signature, BlsScalar)]) -> Vec<bool>   (new)
// Values are held as the reference's wire encodings; every check runs on the GPU.  Header only.
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <optional>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include "jjschnorr_b200.h"

namespace jubjub_schnorr {

enum class Error : uint8_t { InvalidSignature = JJS_INVALID_SIGNATURE, InvalidPoint = JJS_INVALID_POINT, BytesError = JJS_BYTES_ERROR };
using Result = std::optional<Error>;  // std::nullopt == Ok(())
using BlsScalar = std::array<uint8_t, 32>;  // BlsScalar::to_bytes()

inline BlsScalar bls_scalar_from_u64(uint64_t x) {
    BlsScalar b{};
    for (int i = 0; i < 8; i++) b[i] = uint8_t(x >> (8 * i));
    return b;
}

// Owns a jjs_ctx.  One host thread at a time.
class Gpu {
public:
    explicit Gpu(const std::vector<int>& devices = {0}) { init(jjs_init(devices.data(), int(devices.size()), &ctx_), "jjs_init"); }
    // A context that holds at most device_memory_limit bytes of device memory on each device (jjs_init_limited).
    Gpu(const std::vector<int>& devices, size_t device_memory_limit) {
        init(jjs_init_limited(devices.data(), int(devices.size()), device_memory_limit, &ctx_), "jjs_init_limited");
    }
    ~Gpu() { if (ctx_) jjs_destroy(ctx_); }
    Gpu(const Gpu&) = delete;
    Gpu& operator=(const Gpu&) = delete;
    jjs_ctx* ctx() const { return ctx_; }
    void check(int rc, const char* what) const {
        if (rc != JJS_SUCCESS) throw std::runtime_error(std::string(what) + ": " + jjs_last_error(ctx_));
    }
    // NEW: whether all n single (JJS_KIND_SINGLE) or double (JJS_KIND_DOUBLE) items verify, by one random linear combination
    // (jjs_verify_all; a batch with a failing item passes with probability at most 2^-128).  Wire buffers as in the C ABI;
    // seed32: nullptr draws fresh secret weights for every call, 32 given bytes are for tests only.
    bool verify_all(int kind, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg32, size_t n, const uint8_t* seed32 = nullptr) const {
        int ok = 0;
        check(jjs_verify_all(ctx_, kind, pk, sig, msg32, n, seed32, &ok), "jjs_verify_all");
        return ok == 1;
    }
    // NEW: whether every item of every part (any kind, jjs_part as for jjs_verify_mixed with every output field NULL) verifies,
    // by one random linear combination over all parts (jjs_verify_all_mixed); seed32 as for verify_all.
    bool verify_all_mixed(const jjs_part* parts, size_t n_parts, const uint8_t* seed32 = nullptr) const {
        int ok = 0;
        check(jjs_verify_all_mixed(ctx_, parts, n_parts, seed32, &ok), "jjs_verify_all_mixed");
        return ok == 1;
    }
    // NEW: per-item results of every part (jjs_part as for jjs_verify_mixed, outputs included) by one random linear combination
    // per group of consecutive items, the per-item equations only in failing groups (jjs_verify_grouped); seed32 as for
    // verify_all.  Returns the number of items verified one by one.
    uint64_t verify_grouped(const jjs_part* parts, size_t n_parts, const uint8_t* seed32 = nullptr) const {
        uint64_t fallback = 0;
        check(jjs_verify_grouped(ctx_, parts, n_parts, seed32, &fallback), "jjs_verify_grouped");
        return fallback;
    }

private:
    void init(int rc, const char* what) {
        if (rc != JJS_SUCCESS) {
            std::string msg = ctx_ ? jjs_last_error(ctx_) : "allocation failed";
            if (ctx_) jjs_destroy(ctx_);
            ctx_ = nullptr;
            throw std::runtime_error(std::string(what) + ": " + msg);  // no CPU fallback
        }
    }
    jjs_ctx* ctx_ = nullptr;
};

inline Result to_result(uint8_t status) { return status == JJS_OK ? Result{} : Result{Error(status)}; }

template <size_t N>
struct Wire {
    static constexpr size_t SIZE = N;
    std::array<uint8_t, N> bytes{};
    const std::array<uint8_t, N>& to_bytes() const { return bytes; }
    bool operator==(const Wire& o) const { return bytes == o.bytes; }
};

// from_bytes validates like the reference: every point must decode (JubJubAffine::from_bytes), the scalar must be
// canonical.  Throws std::invalid_argument (BytesError::InvalidData) otherwise.
inline void require_points(Gpu& gpu, const uint8_t* pts, size_t n) {
    std::vector<uint8_t> out(n);
    gpu.check(jjs_subgroup_check(gpu.ctx(), pts, n, 0, out.data()), "jjs_subgroup_check");
    for (uint8_t o : out)
        if (o == 0xff) throw std::invalid_argument("BytesError::InvalidData: not a canonical JubJub point");
}
inline void require_scalar(const uint8_t* u) {
    static const uint8_t R_ORDER[32] = {0xb7, 0x2c, 0xf7, 0xd6, 0x5e, 0x0e, 0x97, 0xd0, 0x82, 0x10, 0xc8, 0xcc, 0x93, 0x20, 0x68, 0xa6,
                                        0x00, 0x3b, 0x34, 0x01, 0x01, 0x3b, 0x67, 0x06, 0xa9, 0xaf, 0x33, 0x65, 0xea, 0xb4, 0x7d, 0x0e};
    for (int i = 31; i >= 0; i--) {
        if (u[i] < R_ORDER[i]) return;
        if (u[i] > R_ORDER[i]) break;
    }
    throw std::invalid_argument("BytesError::InvalidData: scalar is not canonical");
}

struct Signature : Wire<64> {
    static Signature from_bytes(Gpu& gpu, const uint8_t* b) {
        Signature s;
        std::memcpy(s.bytes.data(), b, 64);
        require_scalar(b);
        require_points(gpu, b + 32, 1);
        return s;
    }
};
struct SignatureDouble : Wire<96> {
    static SignatureDouble from_bytes(Gpu& gpu, const uint8_t* b) {
        SignatureDouble s;
        std::memcpy(s.bytes.data(), b, 96);
        require_scalar(b);
        require_points(gpu, b + 32, 2);
        return s;
    }
};
struct SignatureVarGen : Wire<64> {
    static SignatureVarGen from_bytes(Gpu& gpu, const uint8_t* b) {
        SignatureVarGen s;
        std::memcpy(s.bytes.data(), b, 64);
        require_scalar(b);
        require_points(gpu, b + 32, 1);
        return s;
    }
};

struct PublicKey : Wire<32> {
    static PublicKey from_bytes(Gpu& gpu, const uint8_t* b) {
        PublicKey k = from_raw_unchecked(b);
        require_points(gpu, b, 1);
        return k;
    }
    static PublicKey from_raw_unchecked(const uint8_t* b) {
        PublicKey k;
        std::memcpy(k.bytes.data(), b, 32);
        return k;
    }
    // reference src/keys/public.rs:114-135
    Result verify(Gpu& gpu, const Signature& sig, const BlsScalar& message) const {
        uint8_t st = 0xff;
        gpu.check(jjs_verify_single(gpu.ctx(), bytes.data(), sig.bytes.data(), message.data(), 1, &st, nullptr), "jjs_verify_single");
        return to_result(st);
    }
    // reference src/keys/public.rs:159-164
    bool is_valid(Gpu& gpu) const {
        static const uint8_t IDENTITY[32] = {1};
        uint8_t out = 0;
        gpu.check(jjs_subgroup_check(gpu.ctx(), bytes.data(), 1, 0, &out), "jjs_subgroup_check");
        return out == 1 && std::memcmp(bytes.data(), IDENTITY, 32) != 0;
    }
};
struct PublicKeyDouble : Wire<64> {
    static PublicKeyDouble from_bytes(Gpu& gpu, const uint8_t* b) {
        PublicKeyDouble k;
        std::memcpy(k.bytes.data(), b, 64);
        require_points(gpu, b, 2);
        return k;
    }
    // reference src/keys/public/double.rs:86-117
    Result verify(Gpu& gpu, const SignatureDouble& sig, const BlsScalar& message) const {
        uint8_t st = 0xff;
        gpu.check(jjs_verify_double(gpu.ctx(), bytes.data(), sig.bytes.data(), message.data(), 1, &st, nullptr), "jjs_verify_double");
        return to_result(st);
    }
};
struct PublicKeyVarGen : Wire<64> {
    static PublicKeyVarGen from_bytes(Gpu& gpu, const uint8_t* b) {
        PublicKeyVarGen k;
        std::memcpy(k.bytes.data(), b, 64);
        require_points(gpu, b, 2);
        return k;
    }
    // reference src/keys/public/var_gen.rs:107-133
    Result verify(Gpu& gpu, const SignatureVarGen& sig, const BlsScalar& message) const {
        uint8_t st = 0xff;
        gpu.check(jjs_verify_vargen(gpu.ctx(), bytes.data(), sig.bytes.data(), message.data(), 1, &st, nullptr), "jjs_verify_vargen");
        return to_result(st);
    }
};

// NEW: verify_batch(&[(PublicKey, Signature, BlsScalar)]) -> Vec<bool>
inline std::vector<bool> verify_batch(Gpu& gpu, const std::vector<std::tuple<PublicKey, Signature, BlsScalar>>& items) {
    const size_t n = items.size();
    std::vector<uint8_t> pk(32 * n), sig(64 * n), msg(32 * n), st(n);
    for (size_t i = 0; i < n; i++) {
        std::memcpy(&pk[32 * i], std::get<0>(items[i]).bytes.data(), 32);
        std::memcpy(&sig[64 * i], std::get<1>(items[i]).bytes.data(), 64);
        std::memcpy(&msg[32 * i], std::get<2>(items[i]).data(), 32);
    }
    if (n) gpu.check(jjs_verify_single(gpu.ctx(), pk.data(), sig.data(), msg.data(), n, st.data(), nullptr), "jjs_verify_single");
    std::vector<bool> out(n);
    for (size_t i = 0; i < n; i++) out[i] = st[i] == JJS_OK;
    return out;
}

namespace multisig {
// reference src/multisig.rs:154-156: sum of d_i * pk_i; the signer keys are not validated
inline PublicKey aggregate_pk(Gpu& gpu, const std::vector<PublicKey>& pk_vec) {
    std::vector<uint8_t> pks(32 * pk_vec.size());
    for (size_t i = 0; i < pk_vec.size(); i++) std::memcpy(&pks[32 * i], pk_vec[i].bytes.data(), 32);
    uint32_t offsets[2] = {0, uint32_t(pk_vec.size())};
    uint8_t sig[64] = {0}, msg[32] = {0}, st = 0, agg[32];
    gpu.check(jjs_verify_aggregate(gpu.ctx(), pks.data(), offsets, sig, msg, 1, &st, nullptr, agg), "jjs_verify_aggregate");
    return PublicKey::from_raw_unchecked(agg);
}
}  // namespace multisig

}  // namespace jubjub_schnorr
