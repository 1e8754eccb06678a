/* rle_oracle.c -- single-threaded C restatement of pycocotools' common/maskApi.c rleEncode + rleToString for one
 * uint8 mask in Fortran (column-major) order, the host cost a caller pays per mask without a device encoder.
 * oracle/rle_oracle.py compiles it on first use and wraps it (CEncoder). */
#include <stdint.h>

/* mask [h*w] column-major, cnts scratch [h*w + 1], s [s_cap]: returns the string length, -1 if s_cap is too small */
int64_t rle_oracle_encode(const uint8_t *M, int64_t h, int64_t w, uint32_t *cnts, char *s, int64_t s_cap) {
    const int64_t a = h * w;
    int64_t j, k = 0, p = 0, i;
    uint32_t c = 0;
    uint8_t prev = 0;
    /* rleEncode */
    for (j = 0; j < a; j++) {
        if (M[j] != prev) {
            cnts[k++] = c;
            c = 0;
            prev = M[j];
        }
        c++;
    }
    cnts[k++] = c;
    /* rleToString */
    for (i = 0; i < k; i++) {
        long x = (long)cnts[i];
        int more = 1;
        if (i > 2) x -= (long)cnts[i - 2];
        while (more) {
            char ch = x & 0x1f;
            x >>= 5;
            more = (ch & 0x10) ? x != -1 : x != 0;
            if (more) ch |= 0x20;
            ch += 48;
            if (p >= s_cap) return -1;
            s[p++] = ch;
        }
    }
    return p;
}
