// emia_coco.cuh — the compressed-RLE "counts" string of COCO instance JSON, as pycocotools' maskApi.c writes and reads it:
//   rleToString: count i (i > 2: its difference to count i - 2) in 5-bit groups, least significant first; a group gets 0x20 when
//     more follow; the loop stops when the rest is 0, or -1 after a group with 0x10 (sign); each group is the character 48 + group;
//   rleFrString: the inverse, a value ending at the first character without 0x20 and sign-extended from its last group's 0x10.
// The alphabet is '0'..'o'; its one character that JSON escapes is '\' (92, a continuation group of value 12), written "\\".
// Compiled into the sm_100a kernels (emia_coco_kernels.cuh) and into tests/hostsim.
#pragma once
#include "emia_common.cuh"

#define EMIA_COCO_MAX_CHARS 7       // a value of more characters is rejected (a count of 32 bits and its delta fit in 7 groups)

EMIA_HD bool emia_coco_char_ok(uint8_t c) { return c >= 48 && c <= 111; }
EMIA_HD bool emia_coco_char_more(uint8_t c) { return ((c - 48) & 0x20) != 0; }

// JSON bytes of delta x (the '\' characters counted twice); *chars (optional) = characters of the counts string
EMIA_HD int emia_coco_delta_len(int64_t x, int* chars) {
    int n = 0, b = 0;
    bool more = true;
    while (more) {
        int c = (int)(x & 0x1f);
        x >>= 5;                                    // arithmetic shift, as the long of maskApi.c
        more = (c & 0x10) ? x != -1 : x != 0;
        if (more) c |= 0x20;
        ++n;
        b += c + 48 == '\\' ? 2 : 1;
    }
    if (chars) *chars = n;
    return b;
}

// the JSON text of delta x at out (emia_coco_delta_len(x) bytes); returns its length
EMIA_HD int emia_coco_put_delta(uint8_t* out, int64_t x) {
    int b = 0;
    bool more = true;
    while (more) {
        int c = (int)(x & 0x1f);
        x >>= 5;
        more = (c & 0x10) ? x != -1 : x != 0;
        if (more) c |= 0x20;
        if (c + 48 == '\\') out[b++] = '\\';
        out[b++] = (uint8_t)(c + 48);
    }
    return b;
}

// the value of the k (1..EMIA_COCO_MAX_CHARS) characters s[0, k) of one rleFrString value, sign-extended from bit 0x10 of the last
EMIA_HD int64_t emia_coco_value(const uint8_t* s, int k) {
    uint64_t x = 0;
    for (int j = 0; j < k; ++j) x |= (uint64_t)((s[j] - 48) & 0x1f) << (5 * j);
    if ((s[k - 1] - 48) & 0x10) x |= ~0ull << (5 * k);
    return (int64_t)x;
}
