// fasta_emul.cpp -- TEST INFRASTRUCTURE.  The contigs FASTA reading of gtsb_parse.cu (kp_fa_*) with
// the stage functions of gt-scaffold_b200/csrc/gtsb_fasta_core.h run as host loops: the whole text
// as one step, lines visited forwards, backwards or in a scrambled order, then the records, the
// length filter and the header sort by rounds over the tied positions, as the device does them.
#include <stdint.h>

#include <algorithm>
#include <numeric>
#include <vector>

#include "../../gt-scaffold_b200/csrc/gtsb_fasta_core.h"

using namespace gtsbf;

extern "C" {

// text: n bytes (8-byte aligned, 8 bytes of room after it).  Returns the IRR_* bits; with 0, the V
// headers in id order (names, off[V + 1]) and seq_len by id.
uint32_t emul_fasta(const char *text, uint64_t n, uint64_t min_len, int order, char *names, uint64_t *off,
                    uint64_t *seq, uint64_t *V) {
  *V = 0;
  std::vector<uint64_t> end;
  for (uint64_t i = 0; i < n; i++)
    if (text[i] == '\n') end.push_back(i + 1);
  if (n && text[n - 1] != '\n') end.push_back(n);
  const uint64_t L = end.size();
  uint32_t irr = 0;
  for (uint64_t i = 0; i < n; i++)
    if (text[i] == 0) irr |= gtsbp::IRR_NUL;
  std::vector<FaLine> line(L);
  for (uint64_t k = 0; k < L; k++) {
    const uint64_t l = order == 0 ? k : order == 1 ? L - 1 - k : (k * 7919) % L;
    if (order > 1 && std::gcd<uint64_t>(7919, L) != 1) continue;
    line[l] = fa_line(text, l ? end[l - 1] : 0, end[l], false, l == 0);
    irr |= line[l].bad;
  }
  if (order > 1 && std::gcd<uint64_t>(7919, L) != 1)
    for (uint64_t l = 0; l < L; l++) {
      line[l] = fa_line(text, l ? end[l - 1] : 0, end[l], false, l == 0);
      irr |= line[l].bad;
    }
  if (irr) return irr;
  std::vector<uint64_t> hs, hl, len;                      // the records: header start, length, seq_len
  for (uint64_t l = 0; l < L; l++) {
    if (line[l].header) {
      hs.push_back((l ? end[l - 1] : 0) + 1);
      hl.push_back(line[l].hlen);
      len.push_back(0);
    } else {
      len.back() += line[l].seq;
    }
  }
  std::vector<uint32_t> klen, kid;
  std::vector<uint64_t> koff;
  std::vector<char> kn;
  for (size_t r = 0; r < hs.size(); r++)
    if (len[r] > min_len) {
      koff.push_back(kn.size());
      kn.insert(kn.end(), text + hs[r], text + hs[r] + hl[r]);
      klen.push_back((uint32_t) hl[r]);
      kid.push_back((uint32_t) r);
    }
  const uint64_t K = klen.size();
  auto key = [&](uint32_t h, uint32_t j) { return fa_key(kn.data() + koff[h], klen[h], j); };
  std::vector<uint32_t> ord(K);
  std::iota(ord.begin(), ord.end(), 0u);
  std::stable_sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return key(a, 0) < key(b, 0); });
  std::vector<uint8_t> bnd(K);
  for (uint64_t p = 0; p < K; p++) bnd[p] = p == 0 || key(ord[p], 0) != key(ord[p - 1], 0);
  std::vector<uint64_t> act(K);
  std::iota(act.begin(), act.end(), 0ull);
  for (uint32_t j = 1; !act.empty(); j++) {
    std::vector<uint64_t> next;
    for (uint64_t p : act)
      if (fa_tied(bnd.data(), p, K)) {
        if (fa_same(bnd.data(), ord.data(), klen.data(), p, j)) return gtsbp::IRR_DUP_NAME;
        next.push_back(p);
      }
    // runs of consecutive tied positions, each sorted by key j
    for (size_t a = 0; a < next.size();) {
      size_t b = a + 1;
      while (b < next.size() && !bnd[next[b]]) b++;
      std::stable_sort(ord.begin() + next[a], ord.begin() + next[b - 1] + 1,
                       [&](uint32_t x, uint32_t y) { return key(x, j) < key(y, j); });
      a = b;
    }
    for (uint64_t p : next)
      if (!bnd[p]) bnd[p] = key(ord[p], j) != key(ord[p - 1], j);
    act.swap(next);
  }
  off[0] = 0;
  for (uint64_t i = 0; i < K; i++) {
    const uint32_t h = ord[i];
    std::copy(kn.begin() + koff[h], kn.begin() + koff[h] + klen[h], names + off[i]);
    off[i + 1] = off[i] + klen[h];
    seq[i] = len[kid[h]];
  }
  *V = K;
  return 0;
}

}
