/*
 * Which of several patterns occur in a file read with fread in 1 MiB blocks and fed to a set match
 * stream (RegexSet::matches, as `grep -f` would ask it); reading stops as soon as the answer is
 * decided, which happens once every pattern has matched.  Prints the index of every matching
 * pattern, one per line.  ANSI C against rure_b200.h:
 *
 *   gcc -ansi -Wall -Werror tests/capi/set_stream.c -Iinclude -Lregex_b200 -lrure_b200 -o set_stream_example
 *   ./set_stream_example big.log 'error' 'timeout' '[0-9]{4}-[0-9]{2}'
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "rure_b200.h"

#define BLOCK (1 << 20)

int main(int argc, char **argv) {
    rure_error *err;
    rure_set *set;
    rure_b200_match_stream *s;
    rure_b200_match_state state;
    const uint8_t **pats;
    size_t *lens, n_pat, i, got;
    uint64_t *mask;
    uint8_t *block;
    FILE *f;
    int ok = 1;

    if (argc < 3) {
        fprintf(stderr, "usage: %s FILE PATTERN...\n", argv[0]);
        return 2;
    }
    n_pat = (size_t)(argc - 2);
    pats = malloc(n_pat * sizeof *pats);
    lens = malloc(n_pat * sizeof *lens);
    mask = calloc((n_pat + 63) / 64, sizeof *mask);
    block = malloc(BLOCK);
    if (pats == NULL || lens == NULL || mask == NULL || block == NULL) {
        fprintf(stderr, "out of memory\n");
        return 1;
    }
    for (i = 0; i < n_pat; i++) {
        pats[i] = (const uint8_t *)argv[i + 2];
        lens[i] = strlen(argv[i + 2]);
    }
    err = rure_error_new();
    set = rure_compile_set(pats, lens, n_pat, RURE_DEFAULT_FLAGS, NULL, err);
    if (set == NULL) {
        fprintf(stderr, "compile: %s\n", rure_error_message(err));
        return 1;
    }
    f = fopen(argv[1], "rb");
    if (f == NULL) {
        perror(argv[1]);
        return 1;
    }
    s = rure_b200_set_match_stream_new(set, 0, 0, 1);
    if (s == NULL) {
        fprintf(stderr, "stream: %s\n", rure_b200_last_error());
        return 1;
    }
    state.decided = 0;
    while (ok && !state.decided && (got = fread(block, 1, BLOCK, f)) > 0)
        ok = rure_b200_match_stream_write(s, block, got) && rure_b200_match_stream_state(s, &state, NULL);
    ok = ok && !ferror(f) && rure_b200_match_stream_finish(s) && rure_b200_match_stream_state(s, &state, mask);
    if (!ok) {
        fprintf(stderr, "stream: %s\n", rure_b200_last_error());
        return 1;
    }
    for (i = 0; i < n_pat; i++)
        if ((mask[i / 64] >> (i % 64)) & 1) printf("%lu\n", (unsigned long)i);
    rure_b200_match_stream_free(s);
    fclose(f);
    free(block);
    free(mask);
    free(lens);
    free(pats);
    rure_set_free(set);
    rure_error_free(err);
    return 0;
}
