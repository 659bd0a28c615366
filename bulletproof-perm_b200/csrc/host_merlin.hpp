// host_merlin.hpp - Merlin 3.0.0 transcripts (STROBE-128 / Keccak-f[1600]) on the host.
//
// Product host code: the Fiat-Shamir transcript stays on the CPU (a few serial sponge calls between
// kernels).  Mirrors merlin::Transcript plus the reference's TranscriptProtocol extension trait
// (/root/reference/bp-perm/src/transcript_protocol.rs:12-68): same method names, same labels, same
// byte framing, so challenges are bit-identical to the Rust crate's.
#pragma once
#include <stdint.h>
#include <string.h>

#include <string>
#include <vector>

namespace bpp_host {

static inline uint64_t rol64(uint64_t v, int n) { return n ? (v << n) | (v >> (64 - n)) : v; }

static inline void keccak_f1600(uint64_t a[25]) {
    static const uint64_t RC[24] = {
        0x0000000000000001ULL, 0x0000000000008082ULL, 0x800000000000808aULL, 0x8000000080008000ULL,
        0x000000000000808bULL, 0x0000000080000001ULL, 0x8000000080008081ULL, 0x8000000000008009ULL,
        0x000000000000008aULL, 0x0000000000000088ULL, 0x0000000080008009ULL, 0x000000008000000aULL,
        0x000000008000808bULL, 0x800000000000008bULL, 0x8000000000008089ULL, 0x8000000000008003ULL,
        0x8000000000008002ULL, 0x8000000000000080ULL, 0x000000000000800aULL, 0x800000008000000aULL,
        0x8000000080008081ULL, 0x8000000000008080ULL, 0x0000000080000001ULL, 0x8000000080008008ULL};
    static const int ROT[5][5] = {{0, 36, 3, 41, 18}, {1, 44, 10, 45, 2}, {62, 6, 43, 15, 61},
                                  {28, 55, 25, 21, 56}, {27, 20, 39, 8, 14}};  // [x][y]
    for (int round = 0; round < 24; round++) {
        uint64_t c[5], d[5], b[25];
        for (int x = 0; x < 5; x++) c[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
        for (int x = 0; x < 5; x++) d[x] = c[(x + 4) % 5] ^ rol64(c[(x + 1) % 5], 1);
        for (int i = 0; i < 25; i++) a[i] ^= d[i % 5];
        for (int x = 0; x < 5; x++)
            for (int y = 0; y < 5; y++) b[y + 5 * ((2 * x + 3 * y) % 5)] = rol64(a[x + 5 * y], ROT[x][y]);
        for (int y = 0; y < 5; y++)
            for (int x = 0; x < 5; x++) a[x + 5 * y] = b[x + 5 * y] ^ (~b[(x + 1) % 5 + 5 * y] & b[(x + 2) % 5 + 5 * y]);
        a[0] ^= RC[round];
    }
}

class Strobe128 {
  public:
    explicit Strobe128(const char *protocol_label) {
        memset(st_, 0, 200);
        const uint8_t init[6] = {1, kR + 2, 1, 0, 1, 96};
        memcpy(st_, init, 6);
        memcpy(st_ + 6, "STROBEv1.0.2", 12);
        permute();
        pos_ = 0;
        pos_begin_ = 0;
        cur_flags_ = 0;
        meta_ad((const uint8_t *)protocol_label, strlen(protocol_label), false);
    }
    // the state of export_state, continued (bpp_transcript_* carry a transcript across the C ABI in this form)
    explicit Strobe128(const uint64_t in[26]) : pos_(0), pos_begin_(0), cur_flags_(0) {
        memset(st_, 0, 200);
        import_state(in);
    }
    void meta_ad(const uint8_t *d, size_t n, bool more) { begin_op(kM | kA, more); absorb(d, n); }
    void ad(const uint8_t *d, size_t n, bool more) { begin_op(kA, more); absorb(d, n); }
    void prf(uint8_t *out, size_t n, bool more) { begin_op(kI | kA | kC, more); squeeze(out, n); }
    // 25 little-endian lanes + pos | pos_begin << 8 | cur_flags << 16: the layout merlin_dev.cuh loads
    void export_state(uint64_t out[26]) const {
        memcpy(out, st_, 200);
        out[25] = (uint64_t)pos_ | ((uint64_t)pos_begin_ << 8) | ((uint64_t)cur_flags_ << 16);
    }
    // false for a word 25 no export could have written (pos, pos_begin beyond the rate, high bits set)
    static bool state_valid(const uint64_t in[26]) {
        const uint64_t w = in[25];
        return !(w >> 24) && (w & 0xff) < kR && ((w >> 8) & 0xff) <= kR;
    }
    // false (state unchanged) if !state_valid(in)
    bool import_state(const uint64_t in[26]) {
        if (!state_valid(in)) return false;
        const uint64_t w = in[25];
        memcpy(st_, in, 200);
        pos_ = (uint8_t)w;
        pos_begin_ = (uint8_t)(w >> 8);
        cur_flags_ = (uint8_t)(w >> 16);
        return true;
    }

  private:
    static const int kR = 166;
    static const uint8_t kI = 1, kA = 2, kC = 4, kM = 16, kK = 32;
    uint8_t st_[200];
    uint8_t pos_, pos_begin_, cur_flags_;
    void permute() {
        uint64_t lanes[25];
        memcpy(lanes, st_, 200);  // little-endian host
        keccak_f1600(lanes);
        memcpy(st_, lanes, 200);
    }
    void run_f() {
        st_[pos_] ^= pos_begin_;
        st_[pos_ + 1] ^= 0x04;
        st_[kR + 1] ^= 0x80;
        permute();
        pos_ = 0;
        pos_begin_ = 0;
    }
    void absorb(const uint8_t *d, size_t n) {
        for (size_t i = 0; i < n; i++) {
            st_[pos_] ^= d[i];
            if (++pos_ == kR) run_f();
        }
    }
    void squeeze(uint8_t *d, size_t n) {
        for (size_t i = 0; i < n; i++) {
            d[i] = st_[pos_];
            st_[pos_] = 0;
            if (++pos_ == kR) run_f();
        }
    }
    void begin_op(uint8_t flags, bool more) {
        if (more) return;  // caller keeps the same flags (merlin asserts this)
        uint8_t old_begin = pos_begin_;
        pos_begin_ = pos_ + 1;
        cur_flags_ = flags;
        uint8_t hdr[2] = {old_begin, flags};
        absorb(hdr, 2);
        if ((flags & (kC | kK)) && pos_ != 0) run_f();
    }
};

// merlin::Transcript + TranscriptProtocol (transcript_protocol.rs)
class Transcript {
  public:
    Transcript(const uint8_t *label, size_t n) : strobe_("Merlin v1.0") { append_message("dom-sep", label, n); }
    explicit Transcript(const uint64_t state[26]) : strobe_(state) {}
    void append_message(const char *label, const uint8_t *msg, size_t n) { append_message(label, strlen(label), msg, n); }
    // labels with an explicit length (merlin's labels are &'static [u8]: any bytes, NUL included)
    void append_message(const char *label, size_t label_len, const uint8_t *msg, size_t n) {
        uint8_t len[4] = {(uint8_t)n, (uint8_t)(n >> 8), (uint8_t)(n >> 16), (uint8_t)(n >> 24)};
        strobe_.meta_ad((const uint8_t *)label, label_len, false);
        strobe_.meta_ad(len, 4, true);
        strobe_.ad(msg, n, false);
    }
    void append_u64(const char *label, uint64_t x) {
        uint8_t b[8];
        for (int i = 0; i < 8; i++) b[i] = (uint8_t)(x >> (8 * i));
        append_message(label, b, 8);
    }
    void challenge_bytes(const char *label, uint8_t *out, size_t n) { challenge_bytes(label, strlen(label), out, n); }
    void challenge_bytes(const char *label, size_t label_len, uint8_t *out, size_t n) {
        uint8_t len[4] = {(uint8_t)n, (uint8_t)(n >> 8), (uint8_t)(n >> 16), (uint8_t)(n >> 24)};
        strobe_.meta_ad((const uint8_t *)label, label_len, false);
        strobe_.meta_ad(len, 4, true);
        strobe_.prf(out, n, false);
    }
    // ---- TranscriptProtocol ----
    void arithmetic_domain_sep(uint64_t n) {  // :27-30
        append_message("dom-sep", (const uint8_t *)"acp v1", 6);
        append_u64("n", n);
    }
    void append_scalar(const char *label, const uint8_t s[32]) { append_message(label, s, 32); }   // :32-34
    void append_point(const char *label, const uint8_t p[32]) { append_message(label, p, 32); }    // :45-47
    bool validate_and_append_point(const char *label, const uint8_t p[32]) {                        // :48-60
        uint8_t o = 0;
        for (int i = 0; i < 32; i++) o |= p[i];
        if (!o) return false;
        append_message(label, p, 32);
        return true;
    }
    // challenge_scalar (:62-67) squeezes 64 bytes; the wide reduction mod l runs on the device
    // (k_scalar_from_wide) or through reduce_wide() below for single values.
    void challenge_wide(const char *label, uint8_t out64[64]) { challenge_bytes(label, out64, 64); }
    void export_state(uint64_t out[26]) const { strobe_.export_state(out); }
    bool import_state(const uint64_t in[26]) { return strobe_.import_state(in); }

  private:
    Strobe128 strobe_;
};

// 512-bit little-endian value mod l on the host (used for single challenges when no launch is worth it)
static inline void reduce_wide(const uint8_t in[64], uint8_t out[32]) {
    // l = 2^252 + c, c = 27742317777372353535851937790883648493; simple long division by repeated shift-subtract
    static const uint32_t Lw[8] = {0x5cf5d3edu, 0x5812631au, 0xa2f79cd6u, 0x14def9deu, 0, 0, 0, 0x10000000u};
    uint32_t r[9] = {0};  // remainder, < 2l
    for (int bit = 511; bit >= 0; bit--) {
        // r = 2r + bit
        uint32_t carry = (in[bit >> 3] >> (bit & 7)) & 1u;
        for (int i = 0; i < 9; i++) {
            uint32_t nc = r[i] >> 31;
            r[i] = (r[i] << 1) | carry;
            carry = nc;
        }
        // if r >= l: r -= l
        uint32_t t[9];
        int64_t borrow = 0;
        for (int i = 0; i < 9; i++) {
            int64_t d = (int64_t)r[i] - (int64_t)(i < 8 ? Lw[i] : 0) + borrow;
            t[i] = (uint32_t)d;
            borrow = d >> 32;
        }
        if (borrow == 0) memcpy(r, t, sizeof(r));
    }
    memcpy(out, r, 32);
}

}  // namespace bpp_host
