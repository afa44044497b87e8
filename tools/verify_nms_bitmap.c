// Algorithm-level replay of nms_kernel phase E for class segments of 1..96 rows (nms.cu): the closed-form work-unit
// layout (seg_units, group-major positions), the suppressor bitmaps built one byte per unit, and the per-warp resolve
// (32 rows per chunk, suppression by kept rows of earlier chunks through the `kept` words, one "ballot" per kept row
// found with ffs) -- against plain greedy NMS on the same overlap relation.  The overlap relation is random with a
// tunable density (clusters), so every segment length and chunk boundary (31/32/33, 63/64/65, 95/96) is hit.
// Both block sizes of nms_kernel (1024 and 512 threads) are replayed: the unit list is walked with the kernel's thread
// stride (every unit exactly once), and the same segment is also resolved by the long-segment path (whole CTA, chunks of
// 32: tests against the kept rows with stride NT, chunk member i on warp i mod NT/32, warp 0's serial resolve).
// usage: verify_nms_bitmap [segments_per_thread]
#include <omp.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define KSHORT 96
static inline uint64_t rng_next(uint64_t* s) {
    uint64_t x = *s;
    x ^= x >> 12;
    x ^= x << 25;
    x ^= x >> 27;
    *s = x;
    return x * 2685821657736338717ULL;
}
static int seg_units(int m) {
    const int G = (m + 6) >> 3;
    return G * (m - 1) - 4 * G * (G - 1);
}

int main(int argc, char** argv) {
    const long per_thread = argc > 1 ? atol(argv[1]) : 200000L;
    long bad = 0, total = 0;
#pragma omp parallel reduction(+ : bad, total)
    {
        uint64_t s = 0x2545F4914F6CDD1DULL * (uint64_t)(omp_get_thread_num() + 7);
        static _Thread_local unsigned char ov[KSHORT][KSHORT];  // ov[j][i], j < i: row j overlaps row i
        for (long it = 0; it < per_thread; ++it) {
            const int m = 1 + (int)(rng_next(&s) % KSHORT);
            const unsigned dens = (unsigned)(rng_next(&s) % 5);  // 0: sparse ... 4: almost everything overlaps
            int cluster[KSHORT];
            for (int i = 0; i < m; ++i) cluster[i] = (int)(rng_next(&s) % (dens == 4 ? 1 : (dens + 2) * 3));
            for (int i = 0; i < m; ++i)
                for (int j = 0; j < i; ++j) {
                    const unsigned r = (unsigned)(rng_next(&s) & 255);
                    ov[j][i] = cluster[i] == cluster[j] ? r < 230 : r < 6 * dens;
                }
            // reference greedy
            unsigned char keep_ref[KSHORT];
            for (int i = 0; i < m; ++i) {
                keep_ref[i] = 1;
                for (int j = 0; j < i; ++j)
                    if (keep_ref[j] && ov[j][i]) {
                        keep_ref[i] = 0;
                        break;
                    }
            }
            // (1a) unit list: row li emits groups g with 8g < li at position off_g + (li - 8g - 1)
            const int U = seg_units(m);
            static _Thread_local int unit_row[KSHORT * 12], unit_g[KSHORT * 12];
            static _Thread_local unsigned char seen[KSHORT * 12];
            memset(seen, 0, (size_t)(U > 0 ? U : 1));
            int layout_ok = 1;
            for (int li = 0; li < m; ++li)
                for (int g = 0; g * 8 < li; ++g) {
                    const int pos = (li - 1) + g * (m - 1) - 4 * g * (g - 1) - 8 * g;
                    if (pos < 0 || pos >= U || seen[pos]) layout_ok = 0;
                    else {
                        seen[pos] = 1;
                        unit_row[pos] = li;
                        unit_g[pos] = g;
                    }
                }
            for (int u = 0; u < U; ++u) layout_ok &= seen[u];
            for (int nt_i = 0; nt_i < 2; ++nt_i) {
            const int NT = nt_i == 0 ? 1024 : 512, NW = NT / 32;
            // (1b) one byte of the row's bitmap per unit; thread tid takes units tid, tid + NT, ...
            unsigned char mask_bytes[KSHORT][12];
            memset(mask_bytes, 0, sizeof(mask_bytes));
            memset(seen, 0, (size_t)(U > 0 ? U : 1));
            for (int tid = 0; tid < NT; ++tid)
                for (int u = tid; u < U; u += NT) seen[u]++;
            for (int u = 0; u < U; ++u) layout_ok &= seen[u] == 1;
            for (int u = 0; u < U && layout_ok; ++u) {
                const int li = unit_row[u], g = unit_g[u];
                unsigned bits = 0;
                for (int k = 0; k < 8; ++k) {
                    const int jx = g * 8 + k;
                    if (jx < li && ov[jx][li]) bits |= 1u << k;
                }
                mask_bytes[li][g] = (unsigned char)bits;
            }
            // (2) resolve, chunks of 32 rows, lanes emulated
            unsigned char keep[KSHORT];
            memset(keep, 0, sizeof(keep));
            unsigned kept[3] = {0, 0, 0};
            for (int c = 0; c < 3; ++c) {
                if (c * 32 >= m) break;
                const int nchunk = m - c * 32 < 32 ? m - c * 32 : 32;
                unsigned mw[32][3];
                unsigned alive = 0;
                for (int lane = 0; lane < 32; ++lane) {
                    mw[lane][0] = mw[lane][1] = mw[lane][2] = 0;
                    if (lane >= nchunk) continue;
                    const int row = c * 32 + lane;
                    for (int w = 0; w <= c; ++w) memcpy(&mw[lane][w], &mask_bytes[row][4 * w], 4);  // little-endian words
                    int removed = 0;
                    for (int w = 0; w < c; ++w) removed |= (mw[lane][w] & kept[w]) != 0u;
                    if (!removed) alive |= 1u << lane;
                }
                for (unsigned rem = alive; rem != 0u;) {
                    const int jx = __builtin_ffs((int)rem) - 1;
                    unsigned kill = 0;
                    for (int lane = 0; lane < 32; ++lane) kill |= ((mw[lane][c] >> jx) & 1u) << lane;  // __ballot_sync
                    alive &= ~kill;
                    rem = alive & ~((2u << jx) - 1u);
                }
                kept[c] = alive;
                for (int lane = 0; lane < 32; ++lane)
                    if ((alive >> lane) & 1u) keep[c * 32 + lane] = 1;
            }
            // (3) the long-segment path on the same segment: chunks of 32 rows against the kept rows so far
            unsigned char keep_long[KSHORT];
            memset(keep_long, 0, sizeof(keep_long));
            int krow[KSHORT], n_kept = 0, members_ok = 1;
            for (int c0 = 0; c0 < m; c0 += 32) {
                const int nchunk = m - c0 < 32 ? m - c0 : 32;
                unsigned rem_bits = 0, sup[32];
                for (int tid = 0; tid < NT; ++tid)
                    for (int p = tid; p < 32 * n_kept; p += NT) {
                        const int i = p & 31, k = p >> 5;
                        if (i < nchunk && ov[krow[k]][c0 + i]) rem_bits |= 1u << i;
                    }
                int written[32] = {0};
                for (int warp = 0; warp < NW; ++warp)
                    for (int i = warp; i < 32; i += NW) {
                        unsigned mm = 0;
                        for (int lane = 0; lane < 32; ++lane)
                            if (i < nchunk && lane < i && ov[c0 + lane][c0 + i]) mm |= 1u << lane;  // __ballot_sync
                        sup[i] = mm;
                        written[i]++;
                    }
                for (int i = 0; i < 32; ++i) members_ok &= written[i] == 1;
                unsigned alive = ~rem_bits & (nchunk == 32 ? 0xffffffffu : ((1u << nchunk) - 1u));
                for (unsigned rem = alive; rem != 0u;) {
                    const int jx = __builtin_ffs((int)rem) - 1;
                    unsigned kill = 0;
                    for (int lane = 0; lane < 32; ++lane) kill |= ((sup[lane] >> jx) & 1u) << lane;
                    alive &= ~kill;
                    rem = alive & ~((2u << jx) - 1u);
                }
                for (int lane = 0; lane < 32; ++lane)
                    if ((alive >> lane) & 1u) {
                        keep_long[c0 + lane] = 1;
                        krow[n_kept++] = c0 + lane;
                    }
            }
            ++total;
            if (!layout_ok || !members_ok || memcmp(keep, keep_ref, (size_t)m) != 0 || memcmp(keep_long, keep_ref, (size_t)m) != 0) {
                ++bad;
                if (bad < 5) printf("MISMATCH NT=%d m=%d dens=%u layout_ok=%d members_ok=%d\n", NT, m, dens, layout_ok, members_ok);
            }
            }
        }
    }
    printf("segments=%ld mismatches=%ld\n", total, bad);
    return bad != 0;
}
