/*
 * memtest_oracle.c — CPU oracle of one march element of the HBM integrity probe (TEST INFRASTRUCTURE).
 * Restates the closed-form pattern of include/b200probe.h independently of the library:
 *   word i of the tested space under seed s = ((uint32_t)i * 2654435761u) ^ s ^ (uint32_t)(i >> 32)
 */
#include <stdint.h>

static uint32_t word_of(uint64_t i, uint32_t seed) { return ((uint32_t)i * 2654435761u) ^ seed ^ (uint32_t)(i >> 32); }

/* words[0..n) hold words base_word.. of the tested space; compare them with the pattern under seed */
void oracle_memtest_verify(const uint32_t* words, uint64_t n, uint64_t base_word, uint32_t seed, uint64_t* bad, uint64_t* first, uint32_t* bits) {
    uint64_t b = 0, f = ~0ull;
    uint32_t x = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const uint32_t want = word_of(base_word + i, seed);
        if (words[i] != want) {
            if (!b) f = base_word + i;
            ++b;
            x |= words[i] ^ want;
        }
    }
    *bad = b; *first = f; *bits = x;
}

/* what an element that writes under seed leaves in words[0..n) */
void oracle_memtest_fill(uint32_t* words, uint64_t n, uint64_t base_word, uint32_t seed) {
    for (uint64_t i = 0; i < n; ++i) words[i] = word_of(base_word + i, seed);
}
