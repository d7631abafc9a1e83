/*
 * Every match of a pattern in a file read with fread in 1 MiB blocks and fed to a
 * rure_b200_stream; the file is never held in memory whole.  Prints one "start end" line per
 * match, then "count N".  PIECE (optional) is the stream's piece size in bytes.  ANSI C against rure_b200.h:
 *
 *   gcc -ansi -Wall -Werror tests/capi/stream.c -Iinclude -Lregex_b200 -lrure_b200 -o stream_example
 *   ./stream_example '[a-zA-Z]+ing' big.log
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "rure_b200.h"

#define BLOCK (1 << 20)
#define SPANS 4096

static int drain(rure_b200_stream *s, rure_match *spans) {
    size_t n, i;
    do {
        if (!rure_b200_stream_read(s, spans, SPANS, &n)) return 0;
        for (i = 0; i < n; i++) printf("%lu %lu\n", (unsigned long)spans[i].start, (unsigned long)spans[i].end);
    } while (n == SPANS);
    return 1;
}

int main(int argc, char **argv) {
    rure_error *err;
    rure *re;
    rure_b200_stream *s;
    FILE *f;
    uint8_t *block;
    rure_match *spans;
    size_t got;
    int ok = 1;

    if (argc != 3 && argc != 4) {
        fprintf(stderr, "usage: %s PATTERN FILE [PIECE]\n", argv[0]);
        return 2;
    }
    err = rure_error_new();
    re = rure_compile((const uint8_t *)argv[1], strlen(argv[1]), RURE_DEFAULT_FLAGS, NULL, err);
    if (re == NULL) {
        fprintf(stderr, "compile: %s\n", rure_error_message(err));
        return 1;
    }
    f = fopen(argv[2], "rb");
    if (f == NULL) {
        perror(argv[2]);
        return 1;
    }
    block = malloc(BLOCK);
    spans = malloc(SPANS * sizeof(rure_match));
    s = rure_b200_stream_new(re, argc == 4 ? strtoul(argv[3], NULL, 10) : 0, 0, 1);
    if (s == NULL || block == NULL || spans == NULL) {
        fprintf(stderr, "stream: %s\n", rure_b200_last_error());
        return 1;
    }
    while (ok && (got = fread(block, 1, BLOCK, f)) > 0)
        ok = rure_b200_stream_write(s, block, got) && drain(s, spans);
    ok = ok && !ferror(f) && rure_b200_stream_finish(s) && drain(s, spans);
    if (!ok) {
        fprintf(stderr, "stream: %s\n", rure_b200_last_error());
        return 1;
    }
    printf("count %lu\n", (unsigned long)rure_b200_stream_count(s));
    rure_b200_stream_free(s);
    free(spans);
    free(block);
    fclose(f);
    rure_free(re);
    rure_error_free(err);
    return 0;
}
