// counts_csv_emu.cpp -- TEST-ONLY: the row decoder of rfx_load_counts_csv (reflexiv_b200/csrc/rfx_counts_csv.cuh) run on the host over a
// whole Count_<k> text, line by line as decode_count_rows_kernel splits it, for comparison with the `reflexiv` binary's parse_counts.
// Not part of libreflexiv_cuda.
#include <cstdint>
#include <cstring>
#include <vector>

#define RFX_NEWLINE_HOSTEMU 1
struct uint4 { uint32_t x, y, z, w; };
#include "../../reflexiv_b200/csrc/rfx_counts_csv.cuh"

using namespace rfx;

extern "C" {
// Kept rows into key_hi / key_lo (the internal right-aligned key split in two words) and counts, at most `cap` of them; returns the
// number of kept rows, or -(line number) of the first malformed row.  The text is copied to a 16-byte aligned buffer whose bytes behind
// the text are ',', '(' and digits: the decoder must not look at them.
int64_t emu_decode_counts(const uint8_t* text, int64_t len, int k, int64_t min_count, int64_t max_count, uint64_t* key_hi, uint64_t* key_lo, uint32_t* counts,
                          int64_t cap) {
    std::vector<uint8_t> buf((size_t)len + 64 + 16);
    uint8_t* t = reinterpret_cast<uint8_t*>(((uintptr_t)buf.data() + 15) & ~(uintptr_t)15);
    memcpy(t, text, (size_t)len);
    for (int i = 0; i < 48; i++) t[len + i] = ",(9)"[i & 3];
    int64_t n = 0, line = 0;
    for (int64_t b = 0; b < len;) {
        const uint8_t* nl = static_cast<const uint8_t*>(memchr(t + b, '\n', (size_t)(len - b)));
        const int64_t e = nl ? nl - t : len;
        line++;
        const CsvRow r = decode_count_row(t, (uint64_t)b, (uint64_t)e, k);
        if (r.kind == CSV_BAD) return -line;
        if (r.kind == CSV_ROW && (int64_t)r.count >= min_count && (int64_t)r.count <= max_count) {
            if (n < cap) {
                key_hi[n] = (uint64_t)(r.key >> 64);
                key_lo[n] = (uint64_t)r.key;
                counts[n] = r.count;
            }
            n++;
        }
        b = e + 1;
    }
    return n;
}
}
