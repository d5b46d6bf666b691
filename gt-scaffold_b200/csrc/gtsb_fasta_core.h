// gtsb_fasta_core.h -- the contigs FASTA read on the device (gtsb_parse.cu, kp_fa_*): the line rule
// and the key of the header sort, one function per stage, so that the same source is the body of the
// kernels and of a plain C++ loop (tests/emul/fasta_emul.cpp).
//
// What is restated: gt_scaffolder_parser_read_contigs (parser.c:420-494) with astat_is_annotated
// false, and the ids of gt_scaffolder_parser_count_distances (the qsort of parser.c:172) --
//   * a record is a line starting with '>' and the sequence lines up to the next such line or the
//     end of the text; the description is the bytes after '>' up to the line's end;
//   * header = the description up to its first ' ', seq_len = the record's sequence bytes;
//   * a record is a vertex iff seq_len > min_ctg_len (parser.c:481);
//   * vertex id = the rank of the header among the vertices' headers in unsigned byte order
//     (strcmp), a header that is a prefix of another first.
// The device accepts the CANONICAL spelling only, on which the stand-in reader, GenomeTools' reader
// and the callbacks cannot disagree: the text starts with '>'; no byte below 0x20 but '\n', none
// equal to 0x7f (a NUL is IRR_NUL, anything else IRR_FASTA); no empty line; a description that is
// not empty and does not start with ' '; sequence lines of [A-Za-z] only; the last line may lack its
// '\n'.  Two vertices with one header are IRR_DUP_NAME (qsort is not stable: the reference's ids are
// unspecified there).
#pragma once
#include <stdint.h>

#include "gtsb_parse_core.h"

namespace gtsbf {

constexpr uint32_t IRR_FASTA = 32u;     // a text outside the canonical FASTA spelling

constexpr uint32_t RADIX_THREADS = 256;
constexpr uint32_t RADIX_ITEMS = 16;                             // consecutive keys per thread
constexpr uint32_t RADIX_TILE = RADIX_THREADS * RADIX_ITEMS;     // keys per block
constexpr uint32_t RADIX_BITS = 4;                               // a pass sorts on 4 key bits
constexpr uint32_t RADIX_BINS = 1u << RADIX_BITS;

struct FaLine {
  uint32_t header;      // 1: a '>' line
  uint32_t hlen;        // header bytes (description up to its first ' ')
  uint32_t seq;         // sequence bytes of the line (no '\n')
  uint32_t bad;         // IRR_FASTA or 0
};

// sequence byte: a letter; a NUL is reported by the newline pass (IRR_NUL) and not here
GTSB_HD bool fa_seq_byte(uint8_t b) {
  const uint8_t l = b | 0x20u;
  return b == 0 || (l >= 'a' && l <= 'z');
}

GTSB_HD bool fa_desc_byte(uint8_t b) { return b == 0 || (b >= 0x20u && b != 0x7fu); }

// eight letters in w: bytes below 0x80, then the case-folded byte in ['a', 'z'] (no carries
// between bytes: l + 0x1f <= 0x9e)
GTSB_HD bool fa_letters8(uint64_t w) {
  const uint64_t H = 0x8080808080808080ull, O = 0x0101010101010101ull;
  if (w & H) return false;
  const uint64_t l = w | (0x20ull * O);
  return ((l + 0x1full * O) & ~(l + 0x05ull * O) & H) == H;
}

// One line [s, e) of a step (e includes its '\n' when it has one).  cont: the line began in an
// earlier step (a sequence line cut at a slot edge); at_start: the first line of the text.
// `t` is 8-byte aligned.
GTSB_HD FaLine fa_line(const char *t, uint64_t s, uint64_t e, bool cont, bool at_start) {
  FaLine f{0u, 0u, 0u, 0u};
  const uint64_t q = e > s && t[e - 1] == '\n' ? e - 1 : e;
  if (!cont && q == s) {                                  // an empty line
    f.bad = IRR_FASTA;
    return f;
  }
  if (!cont && t[s] == '>') {
    f.header = 1u;
    const uint64_t d = s + 1;
    if (d == q || t[d] == ' ') f.bad = IRR_FASTA;         // empty description, or one starting with ' '
    uint64_t h = q;
    for (uint64_t i = d; i < q; i++) {
      const uint8_t b = (uint8_t) t[i];
      if (!fa_desc_byte(b)) f.bad = IRR_FASTA;
      if (b == ' ' && h == q) h = i;
    }
    f.hlen = (uint32_t) (h - d);
    return f;
  }
  if (at_start && !cont) f.bad = IRR_FASTA;               // the text starts with '>'
  f.seq = (uint32_t) (q - s);
  uint64_t i = s;
  for (; i < q && (i & 7u); i++)
    if (!fa_seq_byte((uint8_t) t[i])) f.bad = IRR_FASTA;
  for (; i + 8 <= q; i += 8)
    if (!fa_letters8(*(const uint64_t *) (t + i)))
      for (uint64_t k = i; k < i + 8; k++)
        if (!fa_seq_byte((uint8_t) t[k])) f.bad = IRR_FASTA;
  for (; i < q; i++)
    if (!fa_seq_byte((uint8_t) t[i])) f.bad = IRR_FASTA;
  return f;
}

// ---- the header sort ------------------------------------------------------------------------
// Key j of a header: its bytes [8j, 8j + 8) big-endian, zero-padded.  A canonical header holds no
// NUL, so two headers whose keys 0..j are equal either both end by byte 8(j + 1) -- then they are
// the same header -- or differ in a later key, the shorter one's being 0: key order, key by key,
// is strcmp order, a prefix first.
GTSB_HD uint64_t fa_key(const char *h, uint32_t len, uint32_t j) {
  uint64_t k = 0;
  for (uint32_t i = 0; i < 8; i++) {
    const uint64_t p = 8ull * j + i;
    k = (k << 8) | (p < len ? (uint64_t) (uint8_t) h[p] : 0ull);
  }
  return k;
}

GTSB_HD uint32_t fa_digit(uint64_t key, uint32_t shift) { return (uint32_t) (key >> shift) & (RADIX_BINS - 1u); }

// position p of the order is tied with a neighbour: its group (positions between two boundaries,
// bnd[p] = 1 where p differs from p - 1) holds two or more headers
GTSB_HD bool fa_tied(const uint8_t *bnd, uint64_t p, uint64_t n) { return !bnd[p] || (p + 1 < n && !bnd[p + 1]); }

// p and p - 1 are tied through key j - 1 and both headers end by byte 8j: the same header
GTSB_HD bool fa_same(const uint8_t *bnd, const uint32_t *ord, const uint32_t *len, uint64_t p, uint32_t j) {
  return !bnd[p] && len[ord[p]] <= 8u * j && len[ord[p - 1]] <= 8u * j;
}

}  // namespace gtsbf
