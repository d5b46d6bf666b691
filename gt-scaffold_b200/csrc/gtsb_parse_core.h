// gtsb_parse_core.h -- the `.de` tokeniser, one function per stage, written so
// that the same source is the body of the CUDA kernels (gtsb_parse.cu) and of a
// plain C++ loop (tests/emul/parse_emul.cpp, which lets the token rules be
// checked against the compiled reference without a GPU).
//
// What is restated: the record loop of gt_scaffolder_parser_read_distances,
// parser.c:323-388 --
//   * fgets with a 1024-byte buffer: a physical line is consumed in pieces of at
//     most 1023 characters, each piece handled as a line of its own;
//   * the last character of every piece is dropped (normally the '\n');
//   * tokens are separated by runs of ' '; the first token names the root
//     contig, an unknown root skips the piece;
//   * every token (the first included) that satisfies
//     sscanf("%[^>,],%ld,%ld,%f") == 4 is a record: the header's last character
//     is the orientation ('+' = same), the rest names the partner contig; an
//     unknown partner skips the record;
//   * any other token starting with ';' flips the direction.
//
// The device accepts the CANONICAL spelling of a record only --
//   header ',' ['-'] 1..18 digits ',' 1..18 digits ',' digits ['.' digits*]  <end of token>
// with a distance that fits int32, a pair count that fits uint32 and a standard
// deviation whose decimal -> float conversion is provably the correctly rounded
// one (below).  A token that contains ',' after a non-empty header and is not
// canonical makes the whole file IRREGULAR: nothing is guessed, the caller is
// told to use the host tokeniser (which calls the C library's sscanf).
#pragma once
#include <stdint.h>

#ifndef GTSB_HD
#if defined(__CUDACC__)
#define GTSB_HD __host__ __device__ __forceinline__
#else
#define GTSB_HD inline
#endif
#endif

namespace gtsbp {

constexpr uint32_t PIECE = 1023;        // characters one fgets(line, 1024, file) returns at most
constexpr uint32_t CHUNK = 64;          // bytes per thread in the newline passes
constexpr uint32_t NOT_FOUND = 0xFFFFFFFFu;

// why a file is refused (bit mask)
enum : uint32_t {
  IRR_NUL = 1u,          // a NUL byte (fgets/strlen/strtok stop there)
  IRR_TOKEN = 2u,        // "header,..." that is not a canonical record
  IRR_RANGE = 4u,        // distance outside int32 or pair count outside uint32
  IRR_FLOAT = 8u,        // std_dev with too many digits / too close to a rounding boundary
  IRR_DUP_NAME = 16u,    // two contigs with the same header (bsearch result unspecified)
};

struct NameTable {
  const char *names;        // headers of vertex 0..V-1, concatenated, no terminators
  const uint64_t *off;      // V+1 offsets into names
  uint64_t *slots;          // open addressing: (fingerprint << 32) | (id + 1); 0 = empty
  uint64_t mask;            // capacity - 1 (capacity is a power of two >= 2V)
};

struct Records {
  uint32_t *root, *ctg;
  int32_t *dist;
  float *std_dev;
  uint32_t *num_pairs;
  uint8_t *flags;
};

GTSB_HD void flag_or(uint32_t *flags, uint32_t bit) {
#if defined(__CUDA_ARCH__)
  if ((*(volatile uint32_t *) flags & bit) != bit) atomicOr(flags, bit);
#else
  *flags |= bit;
#endif
}

GTSB_HD uint64_t cas64(uint64_t *addr, uint64_t expect, uint64_t val) {
#if defined(__CUDA_ARCH__)
  return atomicCAS((unsigned long long *) addr, (unsigned long long) expect, (unsigned long long) val);
#else
  const uint64_t old = *addr;
  if (old == expect) *addr = val;
  return old;
#endif
}

// FNV-1a over the bytes, then a 64-bit finaliser so that both the slot index
// (low bits) and the fingerprint (high bits) depend on every byte
GTSB_HD uint64_t hash_bytes(const char *p, uint64_t n) {
  uint64_t h = 0xcbf29ce484222325ull;
  for (uint64_t i = 0; i < n; i++) {
    h ^= (uint8_t) p[i];
    h *= 0x100000001b3ull;
  }
  h ^= h >> 33;
  h *= 0xff51afd7ed558ccdull;
  h ^= h >> 33;
  h *= 0xc4ceb9fe1a85ec53ull;
  h ^= h >> 33;
  return h;
}

GTSB_HD bool same_bytes(const char *a, const char *b, uint64_t n) {
  for (uint64_t i = 0; i < n; i++)
    if (a[i] != b[i]) return false;
  return true;
}

// one vertex into the table; a second contig with the same header is reported
GTSB_HD void table_insert(const NameTable &t, uint32_t v, uint32_t *irregular) {
  const char *name = t.names + t.off[v];
  const uint64_t len = t.off[v + 1] - t.off[v];
  const uint64_t h = hash_bytes(name, len);
  const uint64_t entry = (h & 0xFFFFFFFF00000000ull) | (uint64_t) (v + 1u);
  for (uint64_t s = h & t.mask;; s = (s + 1) & t.mask) {
    const uint64_t old = cas64(t.slots + s, 0ull, entry);
    if (old == 0ull) return;
    if ((old >> 32) == (h >> 32)) {
      const uint32_t u = (uint32_t) old - 1u;
      if (t.off[u + 1] - t.off[u] == len && same_bytes(t.names + t.off[u], name, len)) {
        flag_or(irregular, IRR_DUP_NAME);
        return;
      }
    }
  }
}

// gt_scaffolder_graph_get_vertex (graph.c:187-216): exact match of the header
GTSB_HD uint32_t table_lookup(const NameTable &t, const char *key, uint64_t len) {
  const uint64_t h = hash_bytes(key, len);
  for (uint64_t s = h & t.mask;; s = (s + 1) & t.mask) {
    const uint64_t e = t.slots[s];
    if (e == 0ull) return NOT_FOUND;
    if ((e >> 32) == (h >> 32)) {
      const uint32_t u = (uint32_t) e - 1u;
      if (t.off[u + 1] - t.off[u] == len && same_bytes(t.names + t.off[u], key, len)) return u;
    }
  }
}

// ---- newline passes ---------------------------------------------------------

// 0x80 in every byte of w that equals c, 0 elsewhere (no carries between bytes)
GTSB_HD uint64_t byte_eq_mask(uint64_t w, uint8_t c) {
  const uint64_t x = w ^ (0x0101010101010101ull * c);
  const uint64_t m = 0x7F7F7F7F7F7F7F7Full;
  return ~(((x & m) + m) | x | m);
}

GTSB_HD uint32_t popcount64(uint64_t x) {
#if defined(__CUDA_ARCH__)
  return (uint32_t) __popcll((unsigned long long) x);
#else
  return (uint32_t) __builtin_popcountll(x);
#endif
}

GTSB_HD uint32_t lowest_set(uint64_t x) {                  // x != 0
#if defined(__CUDA_ARCH__)
  return (uint32_t) (__ffsll((long long) x) - 1);
#else
  return (uint32_t) __builtin_ctzll(x);
#endif
}

// '\n' count of chunk i; NUL bytes are reported.  `text` is 8-byte aligned, whole
// words are read as such (little endian: byte j of the word is text[p + j]).
GTSB_HD uint32_t chunk_newlines(const char *text, uint64_t n, uint64_t i, uint32_t *irregular) {
  const uint64_t a = i * CHUNK, b = a + CHUNK < n ? a + CHUNK : n;
  uint32_t c = 0;
  uint64_t nul = 0;
  uint64_t p = a;
  for (; p + 8 <= b; p += 8) {
    const uint64_t w = *(const uint64_t *) (text + p);
    c += popcount64(byte_eq_mask(w, (uint8_t) '\n'));
    nul |= byte_eq_mask(w, 0);
  }
  for (; p < b; p++) {
    c += text[p] == '\n';
    nul |= text[p] == '\0';
  }
  if (nul) flag_or(irregular, IRR_NUL);
  return c;
}

// line_end[r] = offset one past the r-th '\n'; first = number of '\n' before chunk i
GTSB_HD void chunk_line_ends(const char *text, uint64_t n, uint64_t i, uint32_t first, uint64_t *line_end) {
  const uint64_t a = i * CHUNK, b = a + CHUNK < n ? a + CHUNK : n;
  uint64_t p = a;
  for (; p + 8 <= b; p += 8) {
    uint64_t m = byte_eq_mask(*(const uint64_t *) (text + p), (uint8_t) '\n');
    while (m) {
      line_end[first++] = p + (lowest_set(m) >> 3) + 1;
      m &= m - 1;
    }
  }
  for (; p < b; p++)
    if (text[p] == '\n') line_end[first++] = p + 1;
}

// ---- tokens -------------------------------------------------------------------

GTSB_HD bool is_digit(char c) { return c >= '0' && c <= '9'; }

// ['-'] 1..18 digits followed by `stop`; returns the index after `stop`, 0 if not canonical
GTSB_HD uint32_t canonical_int(const char *t, uint32_t i, uint32_t n, bool allow_minus, int64_t *out,
                               char stop = ',') {
  bool neg = false;
  if (allow_minus && i < n && t[i] == '-') {
    neg = true;
    i++;
  }
  uint64_t v = 0;
  uint32_t digits = 0;
  while (i < n && is_digit(t[i])) {
    if (++digits > 18) return 0;
    v = v * 10u + (uint64_t) (t[i] - '0');
    i++;
  }
  if (digits == 0 || i >= n || t[i] != stop) return 0;
  *out = neg ? -(int64_t) v : (int64_t) v;
  return i + 1;
}

// digits ['.' digits*] up to the end of the token.  The value is w / 10^k with
// w the integer spelled by all digits and k the number of digits after the '.'.
//   w <= 2^24, k <= 10: w and 10^k are exact floats, and an IEEE division of two
//       exact operands is the correctly rounded quotient -- what strtof returns;
//   w <= 2^53, k <= 22: the same argument gives the correctly rounded DOUBLE d;
//       the true value lies within half a double ulp of d, so rounding d to float
//       is right unless d sits within one double ulp of the midpoint of two
//       floats -- those (and anything longer) are left to the host's strtof.
// returns 0 ok, IRR_TOKEN (not this spelling) or IRR_FLOAT
GTSB_HD uint32_t canonical_float(const char *t, uint32_t i, uint32_t n, float *out) {
  uint64_t w = 0;
  uint32_t sig = 0, k = 0, int_digits = 0;
  bool dot = false;
  for (; i < n; i++) {
    const char c = t[i];
    if (c == '.') {
      if (dot || int_digits == 0) return IRR_TOKEN;
      dot = true;
      continue;
    }
    if (!is_digit(c)) return IRR_TOKEN;
    if (dot) k++; else int_digits++;
    if (sig > 0 || c != '0') sig++;
    if (sig > 18) return IRR_FLOAT;
    w = w * 10u + (uint64_t) (c - '0');
  }
  if (int_digits == 0) return IRR_TOKEN;
  if (k > 22) return IRR_FLOAT;
  if (w <= (1ull << 24) && k <= 10) {
    float p = 1.0f;
    for (uint32_t j = 0; j < k; j++) p *= 10.0f;
    *out = (float) (uint32_t) w / p;
    return 0;
  }
  if (w > (1ull << 53)) return IRR_FLOAT;
  double p = 1.0;
  for (uint32_t j = 0; j < k; j++) p *= 10.0;
  const double d = (double) w / p;
  union { double f; uint64_t u; } bits;
  bits.f = d;
  const uint64_t low = bits.u & 0x1FFFFFFFull;           // the 29 bits a float does not keep
  if (low >= 0x0FFFFFFFull && low <= 0x10000001ull) return IRR_FLOAT;
  *out = (float) d;
  return 0;
}

struct Token {
  uint32_t ctg;        // partner id or NOT_FOUND
  int32_t dist;
  uint32_t num_pairs;
  float std_dev;
  bool same;
};

// 0: not a record; 1: record (tok filled); otherwise IRR_TOKEN, IRR_RANGE or IRR_FLOAT (all > 1)
GTSB_HD uint32_t parse_token(const char *t, uint32_t n, const NameTable &tab, Token *tok) {
  uint32_t j = 0;
  while (j < n && t[j] != ',' && t[j] != '>') j++;
  // %[^>,] needs one character at least and then a ','; without either sscanf
  // returns 0 or 1 whatever follows
  if (j == 0 || j == n || t[j] != ',') return 0;
  int64_t dist, pairs;
  uint32_t i = canonical_int(t, j + 1, n, true, &dist);
  if (i == 0) return IRR_TOKEN;
  i = canonical_int(t, i, n, false, &pairs);
  if (i == 0) return IRR_TOKEN;
  const uint32_t bad = canonical_float(t, i, n, &tok->std_dev);
  if (bad) return bad;
  if (dist > 2147483647ll || dist < -2147483648ll || pairs > 4294967295ll) return IRR_RANGE;
  tok->dist = (int32_t) dist;
  tok->num_pairs = (uint32_t) pairs;
  tok->same = t[j - 1] == '+';                               // parser.c:347
  tok->ctg = table_lookup(tab, t, j - 1);
  return 1;
}

// One physical line [s, e) (e includes the '\n' when there is one).  EMIT: write
// the records to out[base...]; otherwise only count them.  Returns the count.
template <bool EMIT>
GTSB_HD uint32_t walk_line(const char *text, uint64_t s, uint64_t e, const NameTable &tab,
                           const Records &out, uint64_t base, uint32_t *irregular) {
  uint32_t count = 0;
  for (uint64_t p = s; p < e;) {
    const uint64_t piece_end = p + PIECE < e ? p + PIECE : e;
    const uint64_t q = piece_end - 1;                        // line[strlen(line) - 1] = '\0'
    uint64_t i = p;
    p = piece_end;
    while (i < q && text[i] == ' ') i++;
    if (i == q) continue;                                    // strtok found no token
    uint64_t te = i;
    while (te < q && text[te] != ' ') te++;
    const uint32_t root = table_lookup(tab, text + i, te - i);
    if (root == NOT_FOUND) continue;                         // parser.c: unknown root, next line
    bool sense = true;
    while (i < q) {
      Token tok;
      const uint32_t kind = parse_token(text + i, (uint32_t) (te - i), tab, &tok);
      if (kind == 1) {
        if (tok.ctg != NOT_FOUND) {
          if (EMIT) {
            const uint64_t r = base + count;
            out.root[r] = root;
            out.ctg[r] = tok.ctg;
            out.dist[r] = tok.dist;
            out.std_dev[r] = tok.std_dev;
            out.num_pairs[r] = tok.num_pairs;
            out.flags[r] = (uint8_t) ((sense ? 1u : 0u) | (tok.same ? 2u : 0u));
          }
          count++;
        }
      } else if (kind != 0) {
        flag_or(irregular, kind);
      } else if (text[i] == ';') {
        sense = !sense;
      }
      i = te;
      while (i < q && text[i] == ' ') i++;
      te = i;
      while (te < q && text[te] != ' ') te++;
    }
  }
  return count;
}

// ---- `.astat` lines (algorithms.c:118-149) ------------------------------------------
// fgets pieces as above; every piece must give
//   sscanf("%s\t%ld\t%ld\t%ld\t%f\t%f") == 6      (header, three counts, copy number, a-statistic)
// or the reference stops with an error; a known header gets the two values, the last
// line of a contig wins.  Canonical spelling: header of non-blank characters at the
// start of the line, ONE '\t' between fields, ['-'] 1..18 digits for the counts,
// ['-'] digits ['.' digits*] for the two values (float rule above), nothing after the
// last one.  Everything else -- including what the reference would reject -- is
// IRREGULAR and left to the host loop.

struct AstatLine {
  uint32_t v;             // vertex or NOT_FOUND
  float copy_num, astat;
};

GTSB_HD uint32_t signed_float_field(const char *t, uint32_t i, uint32_t end, float *out) {
  bool neg = false;
  if (i < end && t[i] == '-') {
    neg = true;
    i++;
  }
  const uint32_t bad = canonical_float(t, i, end, out);
  if (bad) return bad;
  if (neg) *out = -*out;
  return 0;
}

// 0 ok, else IRR_* bits
GTSB_HD uint32_t parse_astat_piece(const char *t, uint32_t n, const NameTable &tab, AstatLine *out) {
  uint32_t h = 0;
  while (h < n && t[h] != '\t') {
    const char c = t[h];
    if (c == ' ' || c == '\n' || c == '\v' || c == '\f' || c == '\r') return IRR_TOKEN;
    h++;
  }
  if (h == 0 || h == n) return IRR_TOKEN;
  uint32_t i = h + 1;
  int64_t ignored;
  for (int k = 0; k < 3; k++) {
    i = canonical_int(t, i, n, true, &ignored, '\t');
    if (i == 0) return IRR_TOKEN;
  }
  uint32_t e = i;
  while (e < n && t[e] != '\t') e++;
  if (e == n) return IRR_TOKEN;
  uint32_t bad = signed_float_field(t, i, e, &out->copy_num);
  if (bad) return bad;
  bad = signed_float_field(t, e + 1, n, &out->astat);
  if (bad) return bad;
  out->v = table_lookup(tab, t, h);
  return 0;
}

GTSB_HD void max64(uint64_t *addr, uint64_t val) {
#if defined(__CUDA_ARCH__)
  atomicMax((unsigned long long *) addr, (unsigned long long) val);
#else
  if (*addr < val) *addr = val;
#endif
}

// One physical line [s, e) of a text that starts at file offset `base`.  APPLY = false:
// last[v] = max(file offset + 1) over the pieces naming v; APPLY = true: the piece that holds
// that maximum writes its values.
template <bool APPLY>
GTSB_HD void walk_astat_line_at(const char *text, uint64_t s, uint64_t e, uint64_t base, const NameTable &tab,
                                uint64_t *last, float *astat, float *copy_num, uint32_t *irregular) {
  for (uint64_t p = s; p < e;) {
    const uint64_t piece_end = p + PIECE < e ? p + PIECE : e;
    AstatLine a;
    const uint32_t bad = parse_astat_piece(text + p, (uint32_t) (piece_end - 1 - p), tab, &a);
    if (bad) {
      flag_or(irregular, bad);
    } else if (a.v != NOT_FOUND) {
      if (!APPLY) {
        max64(last + a.v, base + p + 1);
      } else if (last[a.v] == base + p + 1) {
        astat[a.v] = a.astat;                                 // algorithms.c:140-141
        copy_num[a.v] = a.copy_num;
      }
    }
    p = piece_end;
  }
}

// the same for a whole text (offsets are file offsets)
template <bool APPLY>
GTSB_HD void walk_astat_line(const char *text, uint64_t s, uint64_t e, const NameTable &tab, uint64_t *last,
                             float *astat, float *copy_num, uint32_t *irregular) {
  walk_astat_line_at<APPLY>(text, s, e, 0, tab, last, astat, copy_num, irregular);
}

}  // namespace gtsbp
