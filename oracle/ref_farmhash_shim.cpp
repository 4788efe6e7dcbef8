// Thin extern "C" shim over the REFERENCE's vendored FarmHash, compiled in place from
// $YTSAURUS_SOURCE_DIR/contrib/libs/farmhash/farmhash.cc (never copied into this repo).
// Output: oracle/_ref/libfarmhash_ref.so — used only by tests to validate the oracle's
// restatement of the fingerprint functions.
#include <contrib/libs/farmhash/farmhash.h>
#include <cstddef>
#include <cstdint>

extern "C" {
uint64_t ref_fingerprint64(const char* s, size_t n) { return ::util::Fingerprint64(s, n); }
uint64_t ref_fingerprint_u64(uint64_t x) { return ::util::Fingerprint(x); }
uint64_t ref_fingerprint_u128(uint64_t lo, uint64_t hi) { return ::util::Fingerprint(::util::Uint128(lo, hi)); }
uint64_t ref_hash128to64(uint64_t lo, uint64_t hi) { return ::util::Hash128to64(::util::Uint128(lo, hi)); }
}
