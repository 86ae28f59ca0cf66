// TEST INFRASTRUCTURE ONLY: a scorer provider (the C ABI of ctcdecode_b200/scorer.py) that answers from a table of
// recorded language-model scores instead of a KenLM model, so that the scorer-path tests need no KenLM build.
//
// A table (tests/golden/*.lmtab.gz unpacked, written by tests/golden/make_lm_tables.py from the original decoder's Scorer) holds
// the model's order, whether it is character based, its vocabulary, and the conditional log probability
// (natural log, as the Scorer returns it) of every n-gram of `order` words the recorded decodes asked for:
//
//   order 3
//   char_based 0
//   vocab <n>          followed by n lines, one word each
//   ngrams <m>         followed by m lines: <the score's IEEE-754 bits, 16 hex digits> TAB <word> TAB ... <word>
//
// The model path handed to ref_scorer_new / ref_lm_vocabulary is the table's path.  The two hooks turn a label
// prefix into words exactly as the Scorer does (the last `order` words, <s>-padded; a character-based model takes
// every label as one word; the sentence score pads with <s> and appends </s>), score any word outside the
// vocabulary with the Scorer's OOV score, and look everything else up.  An n-gram missing from the table is
// reported on stderr and scored NaN, which no comparison with recorded results survives.
//
// Recording: lm_replay_record(scorer, fn, ctx) installs a source that scores missing n-grams (and stores them);
// lm_replay_save writes the table back.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

namespace {

const double kOovScore = -1000.0;
typedef double (*score_fn)(void *ctx, const char *const *words, int n);

struct Table {
  int order = 0, char_based = 0, space_id = -1;
  std::vector<std::string> vocab, labels;
  std::unordered_set<std::string> known;
  std::unordered_map<std::string, double> scores;  // key: words joined by '\t'
  score_fn source = nullptr;
  void *source_ctx = nullptr;
  std::mutex recording;  // the hooks are called from several threads; only recording writes the table
};

bool read_line(FILE *f, std::string *out) {
  out->clear();
  int c;
  while ((c = fgetc(f)) != EOF && c != '\n') out->push_back(static_cast<char>(c));
  return c != EOF || !out->empty();
}

bool load(const char *path, Table *t) {
  FILE *f = fopen(path, "rb");
  if (!f) return false;
  std::string line;
  size_t n = 0, m = 0;
  bool ok = read_line(f, &line) && sscanf(line.c_str(), "order %d", &t->order) == 1 &&
            read_line(f, &line) && sscanf(line.c_str(), "char_based %d", &t->char_based) == 1 &&
            read_line(f, &line) && sscanf(line.c_str(), "vocab %zu", &n) == 1;
  for (size_t i = 0; ok && i < n; ++i) {
    ok = read_line(f, &line);
    t->vocab.push_back(line);
  }
  ok = ok && read_line(f, &line) && sscanf(line.c_str(), "ngrams %zu", &m) == 1;
  for (size_t i = 0; ok && i < m; ++i) {
    ok = read_line(f, &line);
    size_t tab = line.find('\t');
    ok = ok && tab != std::string::npos;
    if (ok) {  // (bits, not a decimal or hex float: those would be read through the locale)
      uint64_t bits = strtoull(line.substr(0, tab).c_str(), nullptr, 16);
      double v;
      memcpy(&v, &bits, sizeof v);
      t->scores[line.substr(tab + 1)] = v;
    }
  }
  fclose(f);
  for (const std::string &w : t->vocab)
    if (w != "<unk>") t->known.insert(w);  // KenLM's index of <unk> is 0: the Scorer treats it as out of vocabulary
  return ok && t->order > 0;
}

double score_ngram(Table *t, const std::vector<std::string> &words) {
  for (const std::string &w : words)
    if (!t->known.count(w)) return kOovScore;
  std::string key;
  for (size_t i = 0; i < words.size(); ++i) key += (i ? "\t" : "") + words[i];
  std::unique_lock<std::mutex> lock(t->recording, std::defer_lock);
  if (t->source) lock.lock();
  auto it = t->scores.find(key);
  if (it != t->scores.end()) return it->second;
  if (t->source) {
    std::vector<const char *> w;
    for (const std::string &s : words) w.push_back(s.c_str());
    double v = t->source(t->source_ctx, w.data(), static_cast<int>(w.size()));
    t->scores[key] = v;
    return v;
  }
  fprintf(stderr, "lm_replay: n-gram not in the table: [%s]\n", key.c_str());
  return NAN;
}

std::vector<std::string> utf8_chars(const std::string &s) {
  std::vector<std::string> out;
  std::string cur;
  for (char c : s) {
    if ((c & 0xc0) != 0x80 && !cur.empty()) {
      out.push_back(cur);
      cur.clear();
    }
    cur.push_back(c);
  }
  out.push_back(cur);
  return out;
}

}  // namespace

extern "C" {

void *ref_scorer_new(double, double, const char *path, const char *const *labels, int n_labels) {
  Table *t = new Table;
  if (!load(path, t)) {
    fprintf(stderr, "lm_replay: cannot read the table %s\n", path);
    delete t;
    return nullptr;
  }
  for (int i = 0; i < n_labels; ++i) {
    t->labels.emplace_back(labels[i]);
    if (t->labels.back() == " ") t->space_id = i;
  }
  return t;
}
void ref_scorer_free(void *s) { delete static_cast<Table *>(s); }
int ref_scorer_is_character_based(void *s) { return static_cast<Table *>(s)->char_based; }
size_t ref_scorer_max_order(void *s) { return static_cast<size_t>(static_cast<Table *>(s)->order); }
void ref_scorer_reset_params(void *, double, double) {}

// the last `order` words of the prefix, oldest first, <s>-padded when the prefix has fewer
double ref_scorer_cond_from_labels(void *s, const int *labels, int n) {
  Table *t = static_cast<Table *>(s);
  std::vector<std::string> ngram;
  int pos = n;  // labels[0, pos) is what is left of the prefix
  for (int k = 0; k < t->order; ++k) {
    std::string word;
    int start = pos;
    if (t->char_based) {
      start = pos > 0 ? pos - 1 : 0;
    } else {
      while (start > 0 && labels[start - 1] != t->space_id) --start;
    }
    for (int i = start; i < pos; ++i) word += t->labels[labels[i]];
    ngram.insert(ngram.begin(), word);
    if (start == 0) {  // reached the root: pad the missing context
      ngram.insert(ngram.begin(), static_cast<size_t>(t->order - k - 1), "<s>");
      break;
    }
    pos = t->char_based ? start : start - 1;  // (a word-based model skips the space)
  }
  return score_ngram(t, ngram);
}

// the sentence score at read-out: <s> x (order - 1), the words, </s>, summed over windows of `order` words
double ref_scorer_sent_from_labels(void *s, const int *labels, int n) {
  Table *t = static_cast<Table *>(s);
  std::vector<std::string> words;
  if (n > 0) {
    std::string text;
    for (int i = 0; i < n; ++i) text += t->labels[labels[i]];
    if (t->char_based) {
      words = utf8_chars(text);
    } else {
      size_t a = 0;
      for (size_t b; (b = text.find(' ', a)) != std::string::npos; a = b + 1)
        if (b > a) words.push_back(text.substr(a, b - a));
      if (a < text.size()) words.push_back(text.substr(a));
    }
  }
  std::vector<std::string> sent(static_cast<size_t>(words.empty() ? t->order : t->order - 1), "<s>");
  sent.insert(sent.end(), words.begin(), words.end());
  sent.push_back("</s>");
  double score = 0.0;
  for (size_t i = 0; i + t->order <= sent.size(); ++i)
    score += score_ngram(t, std::vector<std::string>(sent.begin() + i, sent.begin() + i + t->order));
  return score;
}

size_t ref_lm_vocabulary(const char *path, char *buf, size_t cap) {
  Table t;
  if (!load(path, &t)) return 0;
  std::string all;
  for (const std::string &w : t.vocab) all += w + "\n";
  if (buf && cap >= all.size() + 1) memcpy(buf, all.c_str(), all.size() + 1);
  return all.size() + 1;
}

void lm_replay_record(void *s, score_fn fn, void *ctx) {
  static_cast<Table *>(s)->source = fn;
  static_cast<Table *>(s)->source_ctx = ctx;
}

int lm_replay_save(void *s, const char *path) {
  Table *t = static_cast<Table *>(s);
  FILE *f = fopen(path, "wb");
  if (!f) return 1;
  fprintf(f, "order %d\nchar_based %d\nvocab %zu\n", t->order, t->char_based, t->vocab.size());
  for (const std::string &w : t->vocab) fprintf(f, "%s\n", w.c_str());
  std::vector<std::string> keys;
  for (const auto &kv : t->scores) keys.push_back(kv.first);
  std::sort(keys.begin(), keys.end());
  fprintf(f, "ngrams %zu\n", keys.size());
  for (const std::string &k : keys) {
    uint64_t bits;
    memcpy(&bits, &t->scores[k], sizeof bits);
    fprintf(f, "%016llx\t%s\n", static_cast<unsigned long long>(bits), k.c_str());
  }
  return fclose(f) != 0;
}

}  // extern "C"
