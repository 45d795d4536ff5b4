/* b200_jit_src.c -- program text of a user QFunction for the NVRTC path of "/gpu/b200:jit" (b200_jit.cu).
 *
 * The locator's file is read as given (absolute, or relative to the current directory; no search path).  Every quoted
 * `#include "..."` whose file exists relative to the including file is inlined in place, recursively, between #line
 * directives, so that NVRTC's messages name the user's file and line.  Angle includes, and quoted ones that do not
 * resolve next to the includer, stay as they are: NVRTC resolves them against its in-memory headers (ceed.h,
 * ceed/ceed.h, math.h) and reports any other as missing.
 */
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "b200_kernels.h"

#define JIT_MAX_DEPTH 32

typedef struct {
  char *p;
  size_t n, cap;
} Buf;

static int buf_put(Buf *b, const char *s, size_t n) {
  if (b->n + n + 1 > b->cap) {
    size_t cap = b->cap ? b->cap : 4096;
    while (b->n + n + 1 > cap) cap *= 2;
    char *q = (char *)realloc(b->p, cap);
    if (!q) return 1;
    b->p = q;
    b->cap = cap;
  }
  memcpy(b->p + b->n, s, n);
  b->n += n;
  b->p[b->n] = 0;
  return 0;
}

static int buf_printf(Buf *b, const char *fmt, ...) {
  char tmp[1200];
  va_list ap;
  va_start(ap, fmt);
  int n = vsnprintf(tmp, sizeof tmp, fmt, ap);
  va_end(ap);
  if (n < 0 || (size_t)n >= sizeof tmp) return 1;
  return buf_put(b, tmp, (size_t)n);
}

static char *read_file(const char *path, size_t *len) {
  FILE *f = fopen(path, "rb");
  if (!f) return NULL;
  Buf b = {0};
  char chunk[8192];
  size_t n;
  while ((n = fread(chunk, 1, sizeof chunk, f)) > 0)
    if (buf_put(&b, chunk, n)) { fclose(f); free(b.p); return NULL; }
  const int bad = ferror(f);
  fclose(f);
  if (bad) { free(b.p); return NULL; }
  if (!b.p && buf_put(&b, "", 0)) return NULL;
  *len = b.n;
  return b.p;
}

/* the quoted file name of `#include "name"` on this line, or 0 */
static int quoted_include(const char *line, const char *end, char *name, size_t cap) {
  const char *s = line;
  while (s < end && (*s == ' ' || *s == '\t')) s++;
  if (s >= end || *s != '#') return 0;
  s++;
  while (s < end && (*s == ' ' || *s == '\t')) s++;
  if ((size_t)(end - s) < 7 || strncmp(s, "include", 7)) return 0;
  s += 7;
  while (s < end && (*s == ' ' || *s == '\t')) s++;
  if (s >= end || *s != '"') return 0;
  const char *q = memchr(s + 1, '"', (size_t)(end - s - 1));
  if (!q || (size_t)(q - s - 1) >= cap || q == s + 1) return 0;
  memcpy(name, s + 1, (size_t)(q - s - 1));
  name[q - s - 1] = 0;
  return 1;
}

/* #line takes a string literal: escape backslashes and quotes of the path */
static int put_line_directive(Buf *out, int line, const char *path) {
  if (buf_printf(out, "#line %d \"", line)) return 1;
  for (const char *c = path; *c; c++) {
    if ((*c == '\\' || *c == '"') && buf_put(out, "\\", 1)) return 1;
    if (buf_put(out, c, 1)) return 1;
  }
  return buf_put(out, "\"\n", 2);
}

static int inline_file(Buf *out, const char *path, int depth, char *err, size_t errlen) {
  if (depth > JIT_MAX_DEPTH) {
    snprintf(err, errlen, "quoted includes nested deeper than %d levels at %s (an include cycle?)", JIT_MAX_DEPTH, path);
    return 1;
  }
  size_t len = 0;
  char *src = read_file(path, &len);
  if (!src) {
    snprintf(err, errlen, "cannot read the QFunction source file \"%s\"", path);
    return 1;
  }
  int rc = put_line_directive(out, 1, path);
  const char *slash = strrchr(path, '/');
  const size_t dirlen = slash ? (size_t)(slash - path + 1) : 0;
  int lineno = 1;
  for (const char *line = src; !rc && line < src + len; lineno++) {
    const char *nl = memchr(line, '\n', (size_t)(src + len - line));
    const char *end = nl ? nl : src + len;
    char name[512], child[1024];
    FILE *probe = NULL;
    if (quoted_include(line, end, name, sizeof name)) {
      if (name[0] == '/') snprintf(child, sizeof child, "%s", name);
      else snprintf(child, sizeof child, "%.*s%s", (int)dirlen, path, name);
      probe = fopen(child, "rb");
    }
    if (probe) {
      fclose(probe);
      rc = inline_file(out, child, depth + 1, err, errlen);
      if (!rc) rc = put_line_directive(out, lineno + 1, path);
    } else {
      rc = buf_put(out, line, (size_t)(end - line));
      if (!rc) rc = buf_put(out, "\n", 1);
    }
    line = nl ? nl + 1 : src + len;
  }
  free(src);
  if (rc && !err[0]) snprintf(err, errlen, "out of memory reading %s", path);
  return rc;
}

int b200_jit_read_source(const char *path, char **text, char *err, size_t errlen) {
  Buf out = {0};
  *text = NULL;
  if (errlen) err[0] = 0;
  if (!path || !path[0]) {
    snprintf(err, errlen, "empty QFunction source path");
    return 1;
  }
  if (inline_file(&out, path, 0, err, errlen)) {
    free(out.p);
    return 1;
  }
  *text = out.p;
  return 0;
}

void b200_jit_free_source(char *text) { free(text); }
