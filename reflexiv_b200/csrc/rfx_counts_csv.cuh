// rfx_counts_csv.cuh -- the per-row arithmetic of rfx_load_counts_csv (rfx_counts_csv.cu): one Count_<k> row (KmerBinarizer input,
// ReflexivDSMain.java:3872-3948) decoded from 16-byte aligned loads of the text.  A header of its own so that tests/hostemu can run the
// same code on the host against the `reflexiv` binary's parse_counts (no CUDA built-ins in here).
#pragma once
#include "rfx_newline.cuh"

namespace rfx {

enum { CSV_SKIP = 0, CSV_ROW = 1, CSV_BAD = 2 };  // an empty line, a row, a malformed row

struct CsvRow {
    unsigned __int128 key;  // the first k characters, 2 bits each, first most significant: the internal (right-aligned) key layout
    uint32_t count;
    uint32_t kind;          // CSV_*
};

// 4 ASCII bytes (first in the low byte) -> 8 bits, first base in bits 7..6.  A=0 C=1 G=2 and every other byte 3, as
// nucleotideValue (ReflexivDSMain.java:3935-3947): 'N' and lower case are 3.
RFX_NL_FN uint32_t csv_encode4(uint32_t w) {
    const uint32_t a = bytes_equal(w, 0x41414141u) >> 7, cc = bytes_equal(w, 0x43434343u) >> 7, g = bytes_equal(w, 0x47474747u) >> 7;
    const uint32_t codes = 0x03030303u - 3u * a - 2u * cc - g;  // one code per byte, no borrow: the three masks are disjoint
    return (codes * 0x40100401u) >> 24;
}

RFX_NL_FN uint32_t csv_word(const uint4& v, uint32_t i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }
RFX_NL_FN uint4 csv_load(const uint8_t* text, uint64_t blk) { return *reinterpret_cast<const uint4*>(text + blk); }
RFX_NL_FN uint32_t csv_byte(const uint8_t* text, uint64_t i) {
    return (csv_word(csv_load(text, i & ~15ull), (uint32_t)(i >> 2) & 3u) >> (8u * (uint32_t)(i & 3))) & 0xffu;
}

// The row on the line [b, e) of `text` (e: its '\n', or the end of the text).  `text` is 16-byte aligned and readable up to the
// 16-byte boundary behind e; bytes outside [b, e) are never used.  The rule of parse_counts (csrc/reflexiv_main.cpp): a trailing '\r'
// is dropped and an empty line skipped; one leading '(' and one trailing ')' are stripped; the k-mer is the first k characters; the
// count is everything behind the first ',': 10 or more characters give 10^9 (ReflexivDSMain.java:3895-3910), fewer are read as
// decimal digits up to the first non-digit.  No ',' or fewer than k characters in front of it: malformed.
RFX_NL_FN CsvRow decode_count_row(const uint8_t* text, uint64_t b, uint64_t e, int k) {
    CsvRow r;
    r.key = 0;
    r.count = 0;
    r.kind = CSV_BAD;
    if (e > b && csv_byte(text, e - 1) == '\r') e--;
    if (b == e) { r.kind = CSV_SKIP; return r; }
    if (csv_byte(text, b) == '(') b++;
    if (e > b && csv_byte(text, e - 1) == ')') e--;
    const uint64_t kend = b + (uint64_t)k;  // the k-mer is [b, kend)
    uint64_t comma = ~0ull, nd = 0;
    bool digits_end = false;
    uint32_t cnt = 0;
    for (uint64_t blk = b & ~15ull; blk < e; blk += 16) {
        const uint4 v = csv_load(text, blk);
        if (blk < kend) {  // bases [lo, hi) of this block belong to the k-mer (1 to 16 of them)
            const uint32_t lo = b > blk ? (uint32_t)(b - blk) : 0u, hi = kend - blk < 16 ? (uint32_t)(kend - blk) : 16u;
            const uint32_t codes = (csv_encode4(v.x) << 24) | (csv_encode4(v.y) << 16) | (csv_encode4(v.z) << 8) | csv_encode4(v.w);
            const uint32_t n = hi - lo;
            r.key = (r.key << (2 * n)) | (uint32_t)((uint32_t)((uint64_t)codes << (2 * lo)) >> (32 - 2 * n));
        }
        if (comma == ~0ull) {
            uint32_t m = mask16(v, 0x2c2c2c2cu);
            if (blk < b) m &= 0xffffu << (uint32_t)(b - blk);
            if (e - blk < 16) m &= (1u << (uint32_t)(e - blk)) - 1u;
            if (!m) continue;
            comma = blk + (uint64_t)lowest_bit(m);
            if (comma < kend) return r;
            nd = e - comma - 1;
            if (nd >= 10) { cnt = 1000000000u; break; }
        }
        // the count's digits in this block: bytes [comma + 1, e), fewer than 10
        const uint64_t from = comma + 1 > blk ? comma + 1 : blk, to = e < blk + 16 ? e : blk + 16;
        for (uint64_t i = from; i < to && !digits_end; i++) {
            const uint32_t ch = (csv_word(v, (uint32_t)(i - blk) >> 2) >> (8u * (uint32_t)(i & 3))) & 0xffu;
            if (ch < '0' || ch > '9') digits_end = true;
            else cnt = cnt * 10u + (ch - '0');
        }
        if (digits_end || e <= blk + 16) break;
    }
    if (comma == ~0ull) return r;
    r.count = cnt;
    r.kind = CSV_ROW;
    return r;
}

}  // namespace rfx
