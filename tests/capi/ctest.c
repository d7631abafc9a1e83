/*
 * The C API test of the Rust `regex` crate (regex-capi/ctest/test.c, MIT OR Apache-2.0),
 * restated: the upstream source is not part of this repository, so its twelve cases are
 * written out here with the upstream patterns, haystacks, lengths (the two size-limit
 * cases pass the pattern with its NUL byte, length 8) and expected values.  It uses
 * nothing but rure.h and is kept to ANSI C, so that it also checks that the header serves
 * strict C90 callers:
 *
 *   gcc -DDEBUG -ansi -Wall -Werror tests/capi/ctest.c -Iinclude -Lregex_b200 -lrure_b200 -o ctest
 *
 * Every case prints "PASSED: <name>" or "FAILED: <name>" on stderr (with -DDEBUG, the
 * reason of a failure too); the exit status is 1 when one failed.
 */
#include <stdbool.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "rure.h"

#ifndef DEBUG
#define DEBUG false
#endif

static bool fail(const char *test, const char *what) {
    if (DEBUG) {
        fprintf(stderr, "[%s] %s\n", test, what);
    }
    return false;
}

static bool same_span(const char *test, rure_match m, size_t start, size_t end) {
    if (m.start != start || m.end != end) {
        if (DEBUG) {
            fprintf(stderr, "[%s] expected (%lu, %lu), got (%lu, %lu)\n", test, (unsigned long)start,
                    (unsigned long)end, (unsigned long)m.start, (unsigned long)m.end);
        }
        return false;
    }
    return true;
}

static bool same_bools(const char *test, const bool *got, const bool *expect, size_t n) {
    size_t i;
    for (i = 0; i < n; ++i) {
        if (got[i] != expect[i]) {
            if (DEBUG) {
                fprintf(stderr, "[%s] pattern %lu: expected %d, got %d\n", test, (unsigned long)i, expect[i], got[i]);
            }
            return false;
        }
    }
    return true;
}

static bool error_says(const char *test, rure_error *err, const char *text) {
    const char *msg = rure_error_message(err);
    if (NULL == strstr(msg, text)) {
        if (DEBUG) {
            fprintf(stderr, "[%s] expected a message with '%s', got '%s'\n", test, text, msg);
        }
        return false;
    }
    return true;
}

bool test_is_match() {
    bool passed = true;
    const char *haystack = "snowman: \xE2\x98\x83";
    rure *re = rure_compile_must("\\p{So}$");
    if (!rure_is_match(re, (const uint8_t *)haystack, strlen(haystack), 0)) {
        passed = fail("test_is_match", "expected match, but got no match");
    }
    rure_free(re);
    return passed;
}

bool test_shortest_match() {
    bool passed = true;
    const char *haystack = "aaaaa";
    size_t end = 0;
    rure *re = rure_compile_must("a+");
    if (!rure_shortest_match(re, (const uint8_t *)haystack, strlen(haystack), 0, &end)) {
        passed = fail("test_shortest_match", "expected match, but got no match");
    } else if (end != 1) {
        passed = fail("test_shortest_match", "expected end 1");
    }
    rure_free(re);
    return passed;
}

bool test_find() {
    bool passed = true;
    const char *haystack = "snowman: \xE2\x98\x83";
    rure_match match = {0};
    rure *re = rure_compile_must("\\p{So}$");
    if (!rure_find(re, (const uint8_t *)haystack, strlen(haystack), 0, &match)) {
        passed = fail("test_find", "expected match, but got no match");
    } else {
        passed = same_span("test_find", match, 9, 12);
    }
    rure_free(re);
    return passed;
}

bool test_captures() {
    bool passed = true;
    const char *haystack = "snowman: \xE2\x98\x83";
    rure_match match = {0};
    rure *re = rure_compile_must(".(.*(?P<snowman>\\p{So}))$");
    rure_captures *caps = rure_captures_new(re);
    if (!rure_find_captures(re, (const uint8_t *)haystack, strlen(haystack), 0, caps)) {
        passed = fail("test_captures", "expected match, but got no match");
    } else if (rure_captures_len(caps) != 3) {
        passed = fail("test_captures", "expected 3 capture groups");
    } else if (rure_capture_name_index(re, "snowman") != 2) {
        passed = fail("test_captures", "expected capture index 2 for 'snowman'");
    } else if (!rure_captures_at(caps, 2, &match)) {
        passed = fail("test_captures", "expected group 2 to take part");
    } else {
        passed = same_span("test_captures", match, 9, 12);
    }
    rure_captures_free(caps);
    rure_free(re);
    return passed;
}

bool test_iter() {
    bool passed = true;
    const uint8_t *haystack = (const uint8_t *)"abc xyz";
    size_t haystack_len = strlen((const char *)haystack);
    rure_match match = {0};
    rure *re = rure_compile_must("\\w+(\\w)");
    rure_captures *caps = rure_captures_new(re);
    rure_iter *it = rure_iter_new(re);
    if (!rure_iter_next(it, haystack, haystack_len, &match)) {
        passed = fail("test_iter", "expected a first match");
    } else if (!same_span("test_iter", match, 0, 3)) {
        passed = false;
    } else if (!rure_iter_next_captures(it, haystack, haystack_len, caps)) {
        passed = fail("test_iter", "expected a second match");
    } else if (!rure_captures_at(caps, 1, &match)) {
        passed = fail("test_iter", "expected group 1 to take part");
    } else {
        passed = same_span("test_iter", match, 6, 7);
    }
    rure_iter_free(it);
    rure_captures_free(caps);
    rure_free(re);
    return passed;
}

bool test_iter_capture_names() {
    bool passed = true;
    static const char *expect[] = {"", "year", "month", "day"};
    char *name = NULL;
    int i;
    rure *re = rure_compile_must("(?P<year>\\d{4})-(?P<month>\\d{2})-(?P<day>\\d{2})");
    rure_iter_capture_names *it = rure_iter_capture_names_new(re);
    for (i = 0; i < 4 && passed; ++i) {
        if (!rure_iter_capture_names_next(it, &name)) {
            passed = fail("test_iter_capture_names", "expected another capture name");
        } else if (strcmp(name, expect[i]) != 0) {
            if (DEBUG) {
                fprintf(stderr, "[test_iter_capture_names] expected '%s', got '%s'\n", expect[i], name);
            }
            passed = false;
        }
    }
    rure_iter_capture_names_free(it);
    rure_free(re);
    return passed;
}

/*
 * No flags at all, which disables Unicode mode: `.` then matches any byte, the invalid
 * UTF-8 byte \xFF included.
 */
bool test_flags() {
    bool passed = true;
    const char *pattern = ".";
    const char *haystack = "\xFF";
    rure *re = rure_compile((const uint8_t *)pattern, strlen(pattern), 0, NULL, NULL);
    if (re == NULL) {
        return fail("test_flags", "expected the pattern to compile");
    }
    if (!rure_is_match(re, (const uint8_t *)haystack, strlen(haystack), 0)) {
        passed = fail("test_flags", "expected match, but got no match");
    }
    rure_free(re);
    return passed;
}

bool test_compile_error() {
    bool passed = true;
    rure_error *err = rure_error_new();
    rure *re = rure_compile((const uint8_t *)"(", 1, 0, NULL, err);
    if (re != NULL) {
        passed = fail("test_compile_error", "expected NULL regex pointer, but got non-NULL pointer");
        rure_free(re);
    }
    if (!error_says("test_compile_error", err, "Unclosed parenthesis")) {
        passed = false;
    }
    rure_error_free(err);
    return passed;
}

bool test_compile_error_size_limit() {
    bool passed = true;
    rure_options *opts = rure_options_new();
    rure_error *err = rure_error_new();
    rure *re;
    rure_options_size_limit(opts, 0);
    re = rure_compile((const uint8_t *)"\\w{100}", 8, 0, opts, err);
    if (re != NULL) {
        passed = fail("test_compile_error_size_limit", "expected NULL regex pointer, but got non-NULL pointer");
        rure_free(re);
    }
    if (!error_says("test_compile_error_size_limit", err, "exceeds size")) {
        passed = false;
    }
    rure_options_free(opts);
    rure_error_free(err);
    return passed;
}

bool test_regex_set_matches() {
    bool passed = true;
    const char *patterns[] = {"foo", "barfoo", "\\w+", "\\d+", "foobar", "bar"};
    const size_t patterns_lengths[] = {3, 6, 3, 3, 6, 3};
    const bool match_target[] = {true, false, true, false, true, true};
    bool matches[6] = {false};
    rure_error *err = rure_error_new();
    rure_set *re = rure_compile_set((const uint8_t **)patterns, patterns_lengths, 6, 0, NULL, err);
    if (re == NULL) {
        passed = fail("test_regex_set_match", "expected the set to compile");
    } else if (rure_set_len(re) != 6) {
        passed = fail("test_regex_set_match", "expected 6 patterns");
    } else if (!rure_set_is_match(re, (const uint8_t *)"foobar", 6, 0)) {
        passed = fail("test_regex_set_match", "expected a match in 'foobar'");
    } else if (rure_set_is_match(re, (const uint8_t *)"", 0, 0)) {
        passed = fail("test_regex_set_match", "expected no match in ''");
    } else if (!rure_set_matches(re, (const uint8_t *)"foobar", 6, 0, matches)) {
        passed = fail("test_regex_set_match", "expected matches in 'foobar'");
    } else {
        passed = same_bools("test_regex_set_match", matches, match_target, 6);
    }
    if (re != NULL) {
        rure_set_free(re);
    }
    rure_error_free(err);
    return passed;
}

bool test_regex_set_options() {
    bool passed = true;
    const char *patterns[] = {"\\w{100}"};
    const size_t patterns_lengths[] = {8};
    rure_options *opts = rure_options_new();
    rure_error *err = rure_error_new();
    rure_set *re;
    rure_options_size_limit(opts, 0);
    re = rure_compile_set((const uint8_t **)patterns, patterns_lengths, 1, 0, opts, err);
    if (re != NULL) {
        passed = fail("test_regex_set_options", "expected NULL regex set pointer, but got non-NULL pointer");
        rure_set_free(re);
    }
    if (!error_says("test_regex_set_options", err, "exceeds size")) {
        passed = false;
    }
    rure_options_free(opts);
    rure_error_free(err);
    return passed;
}

bool test_regex_set_match_start() {
    bool passed = true;
    const char *patterns[] = {"foo", "bar", "fooo"};
    const size_t patterns_lengths[] = {3, 3, 4};
    const bool target_at_0[] = {true, true, true};
    const bool target_at_1[] = {false, true, false};
    bool matches[3] = {false};
    rure_error *err = rure_error_new();
    rure_set *re = rure_compile_set((const uint8_t **)patterns, patterns_lengths, 3, 0, NULL, err);
    if (re == NULL) {
        passed = fail("test_regex_set_match_start", "expected the set to compile");
    } else if (rure_set_len(re) != 3) {
        passed = fail("test_regex_set_match_start", "expected 3 patterns");
    } else if (rure_set_is_match(re, (const uint8_t *)"foobiasdr", 7, 2)) {
        passed = fail("test_regex_set_match_start", "expected no match from offset 2");
    } else if (!rure_set_matches(re, (const uint8_t *)"fooobar", 8, 0, matches)) {
        passed = fail("test_regex_set_match_start", "expected matches from offset 0");
    } else if (!same_bools("test_regex_set_match_start", matches, target_at_0, 3)) {
        passed = false;
    } else if (!rure_set_matches(re, (const uint8_t *)"fooobar", 7, 1, matches)) {
        passed = fail("test_regex_set_match_start", "expected matches from offset 1");
    } else {
        passed = same_bools("test_regex_set_match_start", matches, target_at_1, 3);
    }
    if (re != NULL) {
        rure_set_free(re);
    }
    rure_error_free(err);
    return passed;
}

void run_test(bool (test)(), const char *name, bool *passed) {
    if (!test()) {
        *passed = false;
        fprintf(stderr, "FAILED: %s\n", name);
    } else {
        fprintf(stderr, "PASSED: %s\n", name);
    }
}

int main() {
    bool passed = true;

    run_test(test_is_match, "test_is_match", &passed);
    run_test(test_shortest_match, "test_shortest_match", &passed);
    run_test(test_find, "test_find", &passed);
    run_test(test_captures, "test_captures", &passed);
    run_test(test_iter, "test_iter", &passed);
    run_test(test_iter_capture_names, "test_iter_capture_names", &passed);
    run_test(test_flags, "test_flags", &passed);
    run_test(test_compile_error, "test_compile_error", &passed);
    run_test(test_compile_error_size_limit, "test_compile_error_size_limit", &passed);
    run_test(test_regex_set_matches, "test_regex_set_match", &passed);
    run_test(test_regex_set_options, "test_regex_set_options", &passed);
    run_test(test_regex_set_match_start, "test_regex_set_match_start", &passed);

    if (!passed) {
        exit(1);
    }
    return 0;
}
