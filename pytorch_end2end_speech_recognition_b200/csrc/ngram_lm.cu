// N-gram language model for the fused prefix beam search: the ARPA loader and the device copy of the model (layout and
// lookups: ngram_lm.cuh).  Everything is parsed and validated on the host before the first CUDA call, so a malformed
// file is rejected on a machine without a GPU too; the device memory is allocated once, at create.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iterator>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include "ngram_lm.cuh"

struct b200ctc_ngram_lm {
  int device = -1, V = 0, blank = 0, order = 0;
  long long counts[b200ctc::kMaxLmOrder] = {};
  void* blob = nullptr;   // one device allocation: nodes, unigram row, unigram nodes, word_of
  b200ctc::LmView view{};
};

namespace b200ctc {

namespace {

// One n-gram of the file while it is read: its history node, word (id of the file's word list), numbers.
struct RawNode {
  int parent;   // -1 for a unigram
  int word;
  int depth;
  double p, bo;
};

inline uint64_t key_of(int parent, int word) { return ((uint64_t)(uint32_t)(parent + 1) << 32) | (uint32_t)word; }

bool is_space(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\v' || c == '\f'; }

void split(const char* s, const char* e, std::vector<std::string>* out) {
  out->clear();
  while (s < e) {
    while (s < e && is_space(*s)) ++s;
    const char* t = s;
    while (t < e && !is_space(*t)) ++t;
    if (t > s) out->emplace_back(s, t);
    s = t;
  }
}

// strtod is correctly rounded, so these are the doubles python's float() gives; the whole token must be a number.
bool parse_number(const std::string& tok, double* out) {
  if (tok.empty() || tok.find_first_of("xX") != std::string::npos) return false;   // no hexadecimal floats
  char* end = nullptr;
  const double v = std::strtod(tok.c_str(), &end);
  if (end != tok.c_str() + tok.size() || std::isnan(v)) return false;
  *out = v;
  return true;
}

bool parse_count(const std::string& s, long long* out) {
  if (s.empty() || s.size() > 15) return false;
  long long v = 0;
  for (char c : s) {
    if (c < '0' || c > '9') return false;
    v = v * 10 + (c - '0');
  }
  *out = v;
  return true;
}

struct Model {
  int order = 0;
  long long counts[kMaxLmOrder] = {};
  std::vector<LmNode> nodes;
  std::vector<double> uni_p;
  std::vector<int> uni_node, word_of;
  int bos_state = 0, eos = 0;
};

// Parse and validate; B200CTC_STATUS_INVALID_VALUE on any defect (see b200ctc_ngram_lm_create).
int load_arpa(const char* path, const char* const* symbols, int V, int blank, Model* m) {
  std::ifstream f(path, std::ios::binary);
  if (!f) return B200CTC_STATUS_INVALID_VALUE;
  const std::string text((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  if (f.bad()) return B200CTC_STATUS_INVALID_VALUE;

  std::vector<std::pair<const char*, const char*>> lines;
  for (const char* s = text.data(), *end = text.data() + text.size(); s < end;) {
    const char* e = static_cast<const char*>(std::memchr(s, '\n', end - s));
    if (!e) e = end;
    const char* a = s;
    const char* b = e;
    while (a < b && is_space(*a)) ++a;
    while (b > a && is_space(b[-1])) --b;
    lines.emplace_back(a, b);
    s = e + 1;
  }
  auto line = [&](size_t i) { return std::string(lines[i].first, lines[i].second); };
  size_t li = 0;
  while (li < lines.size() && line(li) != "\\data\\") ++li;   // text before \data\ is ignored
  if (li == lines.size()) return B200CTC_STATUS_INVALID_VALUE;
  ++li;
  // ---- header: "ngram k=count" for k = 1..N ----
  std::vector<long long> declared;
  std::vector<std::string> tok;
  for (; li < lines.size(); ++li) {
    const std::string l = line(li);
    if (l.empty()) {
      if (declared.empty()) continue;
      break;
    }
    if (l.compare(0, 6, "ngram ") != 0) break;
    const size_t eq = l.find('=');
    if (eq == std::string::npos) return B200CTC_STATUS_INVALID_VALUE;
    std::string ks = l.substr(6, eq - 6), cs = l.substr(eq + 1);
    ks.erase(0, ks.find_first_not_of(" \t"));
    ks.erase(ks.find_last_not_of(" \t") + 1);
    cs.erase(0, cs.find_first_not_of(" \t"));
    long long k = 0, c = 0;
    if (!parse_count(ks, &k) || !parse_count(cs, &c)) return B200CTC_STATUS_INVALID_VALUE;
    if (k != (long long)declared.size() + 1 || k > kMaxLmOrder) return B200CTC_STATUS_INVALID_VALUE;
    declared.push_back(c);
  }
  const int N = (int)declared.size();
  if (N < 1) return B200CTC_STATUS_INVALID_VALUE;

  // ---- the n-grams, order by order: words interned in the order the file names them ----
  std::unordered_map<std::string, int> word_id;
  std::vector<RawNode> raw;
  std::unordered_map<uint64_t, int> child;   // (parent node, word) -> node
  long long total = 0;
  for (long long c : declared) total += c;
  if (total > 0x3fffffffLL) return B200CTC_STATUS_INVALID_VALUE;
  raw.reserve((size_t)total);
  child.reserve((size_t)total);
  for (int k = 1; k <= N; ++k) {
    while (li < lines.size() && lines[li].first == lines[li].second) ++li;
    if (li == lines.size() || line(li) != "\\" + std::to_string(k) + "-grams:") return B200CTC_STATUS_INVALID_VALUE;
    ++li;
    for (long long n = 0; n < declared[k - 1]; ++n, ++li) {
      if (li == lines.size()) return B200CTC_STATUS_INVALID_VALUE;
      split(lines[li].first, lines[li].second, &tok);
      // "logp w1 .. wk [bo]"; the highest order carries no back-off weight
      if ((int)tok.size() != k + 1 && !((int)tok.size() == k + 2 && k < N)) return B200CTC_STATUS_INVALID_VALUE;
      RawNode r;
      r.bo = 0.0;
      r.depth = k;
      if (!parse_number(tok[0], &r.p)) return B200CTC_STATUS_INVALID_VALUE;
      if ((int)tok.size() == k + 2 && !parse_number(tok[k + 1], &r.bo)) return B200CTC_STATUS_INVALID_VALUE;
      int parent = -1;
      for (int j = 1; j < k; ++j) {   // the history must itself be an n-gram
        auto w = word_id.find(tok[j]);
        if (w == word_id.end()) return B200CTC_STATUS_INVALID_VALUE;
        auto it = child.find(key_of(parent, w->second));
        if (it == child.end()) return B200CTC_STATUS_INVALID_VALUE;
        parent = it->second;
      }
      auto w = word_id.find(tok[k]);
      if (w == word_id.end()) {
        if (k > 1) return B200CTC_STATUS_INVALID_VALUE;   // a word that is not a unigram
        w = word_id.emplace(tok[k], (int)word_id.size()).first;
      }
      r.parent = parent;
      r.word = w->second;
      if (!child.emplace(key_of(parent, r.word), (int)raw.size()).second) return B200CTC_STATUS_INVALID_VALUE;   // twice
      raw.push_back(r);
    }
    // a section with more lines than its header declares
    if (li < lines.size() && lines[li].first != lines[li].second && lines[li].first[0] != '\\')
      return B200CTC_STATUS_INVALID_VALUE;
  }
  while (li < lines.size() && lines[li].first == lines[li].second) ++li;
  if (li == lines.size() || line(li) != "\\end\\") return B200CTC_STATUS_INVALID_VALUE;

  // ---- symbols -> words ----
  const int BOS = V, EOS = V + 1, UNK = V + 2, NW = lm_n_words(V);
  auto ws = word_id.find("<s>"), we = word_id.find("</s>");
  if (ws == word_id.end() || we == word_id.end()) return B200CTC_STATUS_INVALID_VALUE;
  std::vector<int> lm_word(word_id.size(), -1);   // file word -> LM word; -1: no symbol maps to it (dropped)
  lm_word[ws->second] = BOS;
  lm_word[we->second] = EOS;
  std::unordered_map<std::string, int> seen;
  std::vector<int> word_of(V, -1);
  int unk_file = -1;
  {
    auto wu = word_id.find("<unk>");
    if (wu != word_id.end()) unk_file = wu->second;
  }
  for (int c = 0; c < V; ++c) {
    if (c == blank) continue;
    if (!symbols[c]) return B200CTC_STATUS_INVALID_VALUE;
    const std::string s(symbols[c]);
    if (s == "<s>" || s == "</s>" || !seen.emplace(s, c).second) return B200CTC_STATUS_INVALID_VALUE;
    auto w = word_id.find(s);
    if (w != word_id.end()) {
      lm_word[w->second] = c;
      word_of[c] = c;
    }
  }
  const int unk_word = unk_file >= 0 ? (lm_word[unk_file] >= 0 ? lm_word[unk_file] : UNK) : -1;
  for (int c = 0; c < V; ++c) {
    if (c == blank || word_of[c] >= 0) continue;
    if (unk_word < 0) return B200CTC_STATUS_INVALID_VALUE;   // neither a unigram nor covered by <unk>
    word_of[c] = unk_word;
    lm_word[unk_file] = unk_word;
  }
  if (unk_file >= 0 && lm_word[unk_file] < 0) lm_word[unk_file] = UNK;

  // ---- keep the n-grams all of whose words are mapped (the others can never be queried), renumber ----
  std::vector<int> keep_idx(raw.size(), -1);   // raw node -> final node
  std::vector<int> raw_of(1, -1);              // final node -> raw node (node 0: the empty history)
  std::vector<std::vector<int>> level(N + 1);
  for (size_t i = 0; i < raw.size(); ++i) {
    const RawNode& r = raw[i];
    if (lm_word[r.word] < 0 || (r.parent >= 0 && keep_idx[r.parent] == -2)) {
      keep_idx[i] = -2;
      continue;
    }
    keep_idx[i] = -1;
    level[r.depth].push_back((int)i);
  }
  m->nodes.assign(1, LmNode{0.0, 0.0, -1, 1, 0, 0, 0, 0});
  for (int k = 1; k <= N; ++k) {
    std::vector<int>& lv = level[k];
    // parents are numbered already (lower order); sort by (parent, word)
    std::sort(lv.begin(), lv.end(), [&](int a, int b) {
      const int pa = raw[a].parent < 0 ? 0 : keep_idx[raw[a].parent];
      const int pb = raw[b].parent < 0 ? 0 : keep_idx[raw[b].parent];
      if (pa != pb) return pa < pb;
      return lm_word[raw[a].word] < lm_word[raw[b].word];
    });
    m->counts[k - 1] = (long long)lv.size();
    for (int i : lv) {
      const int id = (int)m->nodes.size();
      keep_idx[i] = id;
      raw_of.push_back(i);
      const int par = raw[i].parent < 0 ? 0 : keep_idx[raw[i].parent];
      LmNode& pn = m->nodes[par];
      if (pn.n_child == 0) pn.first_child = id;
      ++pn.n_child;
      m->nodes.push_back(LmNode{raw[i].p, raw[i].bo, lm_word[raw[i].word], 0, 0, 0, k, 0});
    }
  }
  m->nodes[0].first_child = 1;
  // back-off links: the longest proper suffix that is an n-gram
  std::vector<int> words;
  for (size_t id = 1; id < m->nodes.size(); ++id) {
    words.clear();
    for (int r = raw_of[id]; r >= 0; r = raw[r].parent) words.push_back(raw[r].word);
    std::reverse(words.begin(), words.end());
    int bk = 0;
    for (size_t j = 1; j < words.size() && bk == 0; ++j) {
      int node = -1;
      for (size_t q = j; q < words.size(); ++q) {
        auto it = child.find(key_of(node, words[q]));
        if (it == child.end()) { node = -1; break; }
        node = it->second;
      }
      if (node >= 0) bk = keep_idx[node];
    }
    m->nodes[id].backoff = bk;
  }
  m->order = N;
  m->uni_p.assign(NW, 0.0);
  m->uni_node.assign(NW, -1);
  for (int id = 1; id <= (int)m->counts[0]; ++id) {
    m->uni_p[m->nodes[id].word] = m->nodes[id].p;
    m->uni_node[m->nodes[id].word] = id;
  }
  m->word_of = word_of;
  m->bos_state = N >= 2 ? m->uni_node[BOS] : 0;
  m->eos = EOS;
  return B200CTC_STATUS_SUCCESS;
}

}  // namespace

int ngram_lm_check(const b200ctc_ngram_lm* lm, int V, int blank) {
  if (!lm || lm->V != V || lm->blank != blank) return B200CTC_STATUS_INVALID_VALUE;
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess) {
    cudaGetLastError();
    return B200CTC_STATUS_EXECUTION_FAILED;
  }
  return cur == lm->device ? B200CTC_STATUS_SUCCESS : B200CTC_STATUS_INVALID_VALUE;
}

LmView ngram_lm_view(const b200ctc_ngram_lm* lm) { return lm->view; }

}  // namespace b200ctc

using namespace b200ctc;

extern "C" {

int b200ctc_ngram_lm_create(const char* arpa_path, const char* const* symbols, int V, int blank, int device,
                            b200ctc_ngram_lm** lm) {
  if (!arpa_path || !symbols || !lm || V < 1 || blank < 0 || blank >= V) return B200CTC_STATUS_INVALID_VALUE;
  Model m;
  int st;
  try {
    st = load_arpa(arpa_path, symbols, V, blank, &m);
  } catch (const std::bad_alloc&) {
    return B200CTC_STATUS_EXECUTION_FAILED;
  }
  if (st != B200CTC_STATUS_SUCCESS) return st;

  // ---- the device copy: one allocation ----
  auto al = [](size_t x) { return (x + 255) / 256 * 256; };
  const size_t off_nodes = 0;
  const size_t off_uni_p = off_nodes + al(m.nodes.size() * sizeof(LmNode));
  const size_t off_uni_node = off_uni_p + al(m.uni_p.size() * sizeof(double));
  const size_t off_word_of = off_uni_node + al(m.uni_node.size() * sizeof(int));
  const size_t bytes = off_word_of + al(m.word_of.size() * sizeof(int));
  std::vector<unsigned char> host(bytes, 0);
  std::memcpy(host.data() + off_nodes, m.nodes.data(), m.nodes.size() * sizeof(LmNode));
  std::memcpy(host.data() + off_uni_p, m.uni_p.data(), m.uni_p.size() * sizeof(double));
  std::memcpy(host.data() + off_uni_node, m.uni_node.data(), m.uni_node.size() * sizeof(int));
  std::memcpy(host.data() + off_word_of, m.word_of.data(), m.word_of.size() * sizeof(int));

  int n = 0, prev = -1;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n || cudaGetDevice(&prev) != cudaSuccess) {
    cudaGetLastError();
    return B200CTC_STATUS_EXECUTION_FAILED;   // no CPU fallback: a CUDA device is required
  }
  b200ctc_ngram_lm* h = new (std::nothrow) b200ctc_ngram_lm();
  if (!h) return B200CTC_STATUS_EXECUTION_FAILED;
  void* blob = nullptr;
  const bool ok = cudaSetDevice(device) == cudaSuccess && cudaMalloc(&blob, bytes) == cudaSuccess &&
                  cudaMemcpy(blob, host.data(), bytes, cudaMemcpyHostToDevice) == cudaSuccess;
  cudaSetDevice(prev);
  if (!ok) {
    cudaGetLastError();
    if (blob) cudaFree(blob);
    delete h;
    return B200CTC_STATUS_EXECUTION_FAILED;
  }
  unsigned char* d = static_cast<unsigned char*>(blob);
  h->device = device;
  h->V = V;
  h->blank = blank;
  h->order = m.order;
  std::copy(m.counts, m.counts + kMaxLmOrder, h->counts);
  h->blob = blob;
  h->view.nodes = reinterpret_cast<const LmNode*>(d + off_nodes);
  h->view.uni_p = reinterpret_cast<const double*>(d + off_uni_p);
  h->view.uni_node = reinterpret_cast<const int*>(d + off_uni_node);
  h->view.word_of = reinterpret_cast<const int*>(d + off_word_of);
  h->view.n_words = lm_n_words(V);
  h->view.order = m.order;
  h->view.bos_state = m.bos_state;
  h->view.eos = m.eos;
  *lm = h;
  return B200CTC_STATUS_SUCCESS;
}

int b200ctc_ngram_lm_destroy(b200ctc_ngram_lm* lm) {
  if (!lm) return B200CTC_STATUS_SUCCESS;
  int prev = -1;
  cudaGetDevice(&prev);
  cudaSetDevice(lm->device);
  const cudaError_t e = cudaFree(lm->blob);
  if (prev >= 0) cudaSetDevice(prev);
  cudaGetLastError();
  delete lm;
  return e == cudaSuccess ? B200CTC_STATUS_SUCCESS : B200CTC_STATUS_EXECUTION_FAILED;
}

int b200ctc_ngram_lm_info(const b200ctc_ngram_lm* lm, int* order, long long* counts) {
  if (!lm || !order || !counts) return B200CTC_STATUS_INVALID_VALUE;
  *order = lm->order;
  std::copy(lm->counts, lm->counts + kMaxLmOrder, counts);
  return B200CTC_STATUS_SUCCESS;
}

}  // extern "C"
