/*
 * lcp_kasai.c -- the exact LCP array for the LCP tests (tests/lcp_reference.py compiles and loads it).
 *
 * Kasai, Lee, Arimura, Arikawa, Park (CPM 2001): lcp[0] = 0 and lcp[r] = the longest common prefix of the suffixes
 * sa[r-1] and sa[r], in O(n).  Exact for ANY valid suffix order of the text (proper prefixes first, sentinel unique or
 * not): the h - 1 carried to suffix i + 1 holds because prepending one symbol to two adjacent suffixes that share it
 * keeps them adjacent.  Independent of the library: plain sequential C over host arrays.
 */
#include <stdint.h>
#include <stdlib.h>

int lcp_kasai(const uint8_t *t, uint64_t n, const uint32_t *sa, uint32_t *lcp)
{
    if (n == 0) return 0;
    uint32_t *rank = (uint32_t *)malloc(n * sizeof(uint32_t));
    if (!rank) return -1;
    for (uint64_t r = 0; r < n; ++r) rank[sa[r]] = (uint32_t)r;
    uint64_t h = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const uint32_t r = rank[i];
        if (r == 0) { lcp[0] = 0; h = 0; continue; }
        const uint64_t j = sa[r - 1];
        while (i + h < n && j + h < n && t[i + h] == t[j + h]) ++h;
        lcp[r] = (uint32_t)h;
        if (h) --h;
    }
    free(rank);
    return 0;
}
