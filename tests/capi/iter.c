/*
 * The iterator example of the Rust `regex` crate's C API (regex-capi/examples/iter.c,
 * MIT OR Apache-2.0), restated (the upstream source is not part of this repository):
 * every match of `(\w+)\s+Holmes` (case-insensitive) in sherlock.txt of the working
 * directory, with the span of the whole match and the text of group 1, then the number of
 * matches.  ANSI C against rure.h:
 *
 *   gcc -ansi -Wall -Werror tests/capi/iter.c -Iinclude -Lregex_b200 -lrure_b200 -o iter_example
 */
#define _POSIX_C_SOURCE 200112L
#include <fcntl.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "rure.h"

int main() {
    const char *pattern = "(\\w+)\\s+Holmes";
    struct stat buf;
    size_t len, n = 0;
    char *data;
    rure_error *err;
    rure *re;
    rure_match match = {0};
    rure_captures *caps;
    rure_iter *it;

    int fd = open("sherlock.txt", O_RDONLY);
    if (fd == -1) {
        perror("failed to open sherlock.txt");
        exit(1);
    }
    if (fstat(fd, &buf) == -1) {
        perror("failed to stat sherlock.txt");
        exit(1);
    }
    len = (size_t)buf.st_size;
    data = mmap(NULL, len, PROT_READ, MAP_PRIVATE, fd, 0);
    if (data == MAP_FAILED) {
        perror("failed to mmap sherlock.txt");
        exit(1);
    }

    err = rure_error_new();
    re = rure_compile((const uint8_t *)pattern, strlen(pattern), RURE_FLAG_UNICODE | RURE_FLAG_CASEI, NULL, err);
    if (NULL == re) {
        fprintf(stderr, "compilation of %s failed: %s\n", pattern, rure_error_message(err));
        exit(1);
    }
    caps = rure_captures_new(re);
    it = rure_iter_new(re);
    while (rure_iter_next_captures(it, (const uint8_t *)data, len, caps)) {
        /* both groups take part in every match of this pattern */
        rure_captures_at(caps, 0, &match);
        printf("match at %lu..%lu: ", (unsigned long)match.start, (unsigned long)match.end);
        rure_captures_at(caps, 1, &match);
        printf("%.*s\n", (int)(match.end - match.start), data + match.start);
        ++n;
    }
    printf("%lu matches\n", (unsigned long)n);

    rure_iter_free(it);
    rure_captures_free(caps);
    rure_free(re);
    rure_error_free(err);
    munmap(data, len);
    close(fd);
    return 0;
}
