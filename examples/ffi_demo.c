/* ffi_demo.c — a host program that uses ONLY include/frz_cuda.h (plain C, no CUDA headers, no Python, no torch):
 * the same calls a Rust `extern "C"` binding makes (INTEGRATION.md §2).
 *
 *   gcc -std=c11 -Iinclude examples/ffi_demo.c -Lfrizbee_b200 -lfrz_cuda -Wl,-rpath,$PWD/frizbee_b200 -o ffi_demo
 *   ./ffi_demo            # BASELINE.json configs[0]: needle "fBr" vs 5 haystacks → [Match{score 53, index 0}]
 *
 *   ./ffi_demo 2          # additionally: match_list_parallel over 2 GPUs (frz_comm_create_local + frz_match_list_parallel)
 *                         # must equal match_list on one GPU (src/matcher/parallel.rs:104-130: parallel == sequential)
 *
 * Exit code 0: matched and printed; 3: no CUDA device (the library never falls back to the CPU); 4: parallel != sequential. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "frz_cuda.h"

/* Matcher::match_list_parallel through the C ABI: a list of `n` generated haystacks, sharded over `n_gpus` GPUs of this
 * process, against the same list on one GPU.  Returns 0 when the two results are identical. */
static int parallel_demo(int n_gpus) {
    enum { N = 100003, MAXLEN = 24 };   /* not a multiple of the GPU count: the last shard is short */
    uint8_t* bytes = malloc((size_t)N * MAXLEN);
    uint32_t* offsets = malloc(((size_t)N + 1) * sizeof *offsets);   /* Arrow Utf8: 32-bit offsets */
    frz_match* seq = malloc((size_t)N * sizeof *seq);
    if (!bytes || !offsets || !seq) return 1;
    uint64_t x = 0x9E3779B97F4A7C15ull;
    uint32_t pos = 0;
    static const char alpha[] = "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789_-/";
    for (int i = 0; i < N; i++) {
        offsets[i] = pos;
        x ^= x << 13; x ^= x >> 7; x ^= x << 17;
        const int len = 6 + (int)(x % (MAXLEN - 6));
        for (int k = 0; k < len; k++) { x ^= x << 13; x ^= x >> 7; x ^= x << 17; bytes[pos + k] = (uint8_t)alpha[x % (sizeof alpha - 1)]; }
        if (i % 7 == 0) memcpy(bytes + pos + (x % 3), "foo", 3);            /* plant matches ...                */
        if (i % 2048 == 0 || i % 2048 == 2047) memcpy(bytes + pos, "foo", 3); /* ... also right at shard/tile seams */
        pos += (uint32_t)len;
    }
    offsets[N] = pos;

    frz_config cfg;
    frz_config_default(&cfg);
    cfg.max_typos = 1;
    frz_pattern pat;
    memset(&pat, 0, sizeof pat);
    pat.needle = (const uint8_t*)"foo";
    pat.needle_len = 3;
    pat.casing = -1; pat.unicode = -1; pat.matching = -1; pat.max_typos = -1;
    frz_matcher* m = NULL;
    frz_corpus* whole = NULL;
    frz_comm* comm = NULL;
    frz_corpus* shards[64] = {0};
    frz_match* par = NULL;
    uint64_t n_seq = 0, n_par = 0;
    int rc = 1;
    frz_status st = frz_matcher_create(&pat, 1, &cfg, &m);
    if (st == FRZ_OK) st = frz_corpus_create_arrow(bytes, offsets, 4, N, 0, &whole);
    if (st == FRZ_OK) st = frz_match_list(m, whole, seq, N, &n_seq);                       /* sequential, one GPU */
    if (st == FRZ_OK) st = frz_comm_create_local(n_gpus, NULL, &comm);                     /* threads -> GPUs */
    if (st == FRZ_OK) st = frz_corpus_create_sharded(bytes, offsets, 4, N, comm, shards);  /* contiguous index ranges */
    if (st == FRZ_OK) st = frz_comm_host_alloc(comm, (uint64_t)N * sizeof(frz_match), (void**)&par);   /* pinned: all GPUs copy at once */
    if (st == FRZ_OK) st = frz_match_list_parallel(m, (const frz_corpus* const*)shards, n_gpus, comm, par, N, &n_par);
    if (st != FRZ_OK) {
        fprintf(stderr, "parallel demo: %s: %s\n", frz_status_str(st), frz_last_error());
    } else {
        const int same = n_seq == n_par && memcmp(seq, par, (size_t)n_seq * sizeof *seq) == 0;
        const int mode = frz_comm_exchange_mode(comm);
        printf("match_list_parallel over %d GPU(s): %llu matches, parallel == sequential: %s (exchange: %s)\n", n_gpus, (unsigned long long)n_par,
               same ? "yes" : "NO", n_gpus == 1 ? "n/a" : mode == 2 ? "P2P placement over NVLink" : "ncclAllGather + merge");
        rc = same ? 0 : 4;
    }
    for (int g = 0; g < 64; g++) frz_corpus_destroy(shards[g]);
    if (comm && par) frz_comm_host_free(comm, par);
    frz_comm_destroy(comm);
    frz_corpus_destroy(whole);
    frz_matcher_destroy(m);
    free(bytes); free(offsets); free(seq);
    return rc;
}

int main(int argc, char** argv) {
    static const char* hay[] = {"fooBar", "foo_bar", "barfoo", "prelude", "println!"};
    enum { N = 5 };
    /* Arrow-style buffers: concatenated bytes + offsets */
    uint8_t bytes[256];
    uint64_t offsets[N + 1] = {0};
    for (int i = 0; i < N; i++) {
        size_t len = strlen(hay[i]);
        memcpy(bytes + offsets[i], hay[i], len);
        offsets[i + 1] = offsets[i] + len;
    }
    printf("frz ABI version %u\n", frz_abi_version());

    frz_config cfg;
    frz_config_default(&cfg);
    cfg.max_typos = 0;

    frz_pattern pat;
    memset(&pat, 0, sizeof pat);
    pat.needle = (const uint8_t*)"fBr";
    pat.needle_len = 3;
    pat.casing = -1; pat.unicode = -1; pat.matching = -1; pat.max_typos = -1;   /* inherit from the config */

    frz_matcher* m = NULL;
    frz_status st = frz_matcher_create(&pat, 1, &cfg, &m);
    if (st != FRZ_OK) { fprintf(stderr, "matcher: %s: %s\n", frz_status_str(st), frz_last_error()); return 1; }

    frz_corpus* corpus = NULL;
    st = frz_corpus_create(bytes, offsets, N, /*device=*/0, &corpus);
    if (st != FRZ_OK) {
        fprintf(stderr, "corpus: %s: %s\n", frz_status_str(st), frz_last_error());
        frz_matcher_destroy(m);
        return st == FRZ_ERR_NO_DEVICE || st == FRZ_ERR_CUDA ? 3 : 1;
    }

    frz_match out[N];
    uint64_t n_out = 0;
    st = frz_match_list(m, corpus, out, N, &n_out);
    if (st != FRZ_OK) { fprintf(stderr, "match_list: %s: %s\n", frz_status_str(st), frz_last_error()); return 1; }
    for (uint64_t i = 0; i < n_out; i++)
        printf("Match { score: %u, index: %u, exact: %s }  \"%s\"\n", out[i].score, out[i].index, out[i].exact ? "true" : "false",
               hay[out[i].index]);

    /* matched character offsets of the displayed rows (Matcher::match_list_indices) */
    uint32_t which[1] = {0}, idx[16], cnt[1];
    frz_match mi[1];
    st = frz_match_indices(m, corpus, which, 1, mi, idx, 16, cnt);
    if (st == FRZ_OK && cnt[0] != UINT32_MAX) {
        printf("indices of \"%s\":", hay[0]);
        for (uint32_t k = 0; k < cnt[0]; k++) printf(" %u", idx[k]);
        printf("\n");
    }
    frz_corpus_destroy(corpus);
    frz_matcher_destroy(m);
    if (argc > 1) return parallel_demo(atoi(argv[1]));
    return 0;
}
