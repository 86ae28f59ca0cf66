// TEST INFRASTRUCTURE ONLY -- not part of the product; nothing under ctcdecode_b200/ links this.
//
// Plain C-ABI driver over the UNMODIFIED reference sources (compiled where they lie under
// /root/reference by oracle/Makefile into oracle/_ref/libctcref.so).  It performs exactly the
// marshalling of the reference's pybind boundary so that tests and bench.py can call the
// reference without torch's C++ ABI:
//   * inputs  : float [B,T,V] -> vector<vector<vector<double>>> clamped to min(seq_len,T)
//               (reference binding.cpp:59-74)
//   * decode  : ctc_beam_search_decoder_batch (reference ctc_beam_search_decoder.cpp:245-285)
//   * outputs : only [b,p,:len] of tokens/timesteps, scores[b,p]=float(first), lens[b,p]
//               are written (reference binding.cpp:79-99)
// and the streaming variant (binding.cpp:153-229, ctc_beam_search_decoder.cpp:288-317).
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "ctc_beam_search_decoder.h"
#include "scorer.h"

namespace {
std::vector<std::string> to_vocab(const char *const *labels, int n) {
  std::vector<std::string> v;
  for (int i = 0; i < n; ++i) v.emplace_back(labels[i]);
  return v;
}
std::vector<std::vector<std::vector<double>>> widen(const float *probs, const int *seq_lens, int B, int T,
                                                   int V) {
  std::vector<std::vector<std::vector<double>>> inputs;
  for (int b = 0; b < B; ++b) {
    int len = std::min(seq_lens[b], T);
    if (len < 0) len = 0;
    std::vector<std::vector<double>> temp(len, std::vector<double>(V));
    for (int t = 0; t < len; ++t)
      for (int n = 0; n < V; ++n) temp[t][n] = probs[(static_cast<size_t>(b) * T + t) * V + n];
    inputs.push_back(std::move(temp));
  }
  return inputs;
}
}  // namespace

extern "C" {

void *ref_scorer_new(double alpha, double beta, const char *lm_path, const char *const *labels, int V) {
  return new Scorer(alpha, beta, lm_path, to_vocab(labels, V));
}
void ref_scorer_free(void *s) { delete static_cast<Scorer *>(s); }
int ref_scorer_is_character_based(void *s) { return static_cast<Scorer *>(s)->is_character_based(); }
size_t ref_scorer_max_order(void *s) { return static_cast<Scorer *>(s)->get_max_order(); }
size_t ref_scorer_dict_size(void *s) { return static_cast<Scorer *>(s)->get_dict_size(); }
void ref_scorer_reset_params(void *s, double a, double b) { static_cast<Scorer *>(s)->reset_params(a, b); }

// Returns 1 like the reference's beam_decode.  n_results[b] additionally reports how many rows p
// the reference wrote for utterance b (rows beyond that are untouched, as in the reference).
int ref_decode_batch(const float *probs, const int *seq_lens, int B, int T, int V, const char *const *labels,
                     size_t beam_size, size_t num_processes, double cutoff_prob, size_t cutoff_top_n,
                     size_t blank_id, int log_input, void *scorer, int *out_tokens, int *out_timesteps,
                     float *out_scores, int *out_lens, int *n_results) {
  auto vocab = to_vocab(labels, V);
  auto inputs = widen(probs, seq_lens, B, T, V);
  auto results = ctc_beam_search_decoder_batch(inputs, vocab, beam_size, num_processes, cutoff_prob,
                                               cutoff_top_n, blank_id, log_input,
                                               static_cast<Scorer *>(scorer));
  for (size_t b = 0; b < results.size(); ++b) {
    const auto &res = results[b];
    if (n_results) n_results[b] = static_cast<int>(res.size());
    for (size_t p = 0; p < res.size(); ++p) {
      const Output &o = res[p].second;
      size_t base = (b * beam_size + p) * static_cast<size_t>(T);
      for (size_t t = 0; t < o.tokens.size(); ++t) {
        out_tokens[base + t] = o.tokens[t];
        out_timesteps[base + t] = o.timesteps[t];
      }
      out_scores[b * beam_size + p] = static_cast<float>(res[p].first);
      out_lens[b * beam_size + p] = static_cast<int>(o.tokens.size());
    }
  }
  return 1;
}

void *ref_state_new(const char *const *labels, int V, size_t beam_size, double cutoff_prob, size_t cutoff_top_n,
                    size_t blank_id, int log_input, void *scorer) {
  return new DecoderState(to_vocab(labels, V), beam_size, cutoff_prob, cutoff_top_n, blank_id, log_input,
                          static_cast<Scorer *>(scorer));
}
void ref_state_free(void *s) { delete static_cast<DecoderState *>(s); }

// Streaming step.  Outputs are written into caller buffers shaped [B, max_results, max_len];
// *res_dims = {max_result_size, max_output_tokens_size} as computed by the reference
// (binding.cpp:181-199).  Tokens beyond a beam's length are left untouched.
int ref_decode_with_states(const float *probs, const int *seq_lens, int B, int T, int V, size_t num_processes,
                           void **states, const uint8_t *is_eos, int max_results_cap, int max_len_cap,
                           int *out_tokens, int *out_timesteps, float *out_scores, int *out_lens,
                           int beam_stride, int *res_dims) {
  auto inputs = widen(probs, seq_lens, B, T, V);
  std::vector<void *> st(states, states + B);
  std::vector<bool> eos(B);
  for (int b = 0; b < B; ++b) eos[b] = is_eos[b] != 0;
  auto results = ctc_beam_search_decoder_batch_with_states(inputs, num_processes, st, eos);
  int max_res = 0, max_len = 0;
  for (auto &res : results) {
    max_res = std::max<int>(max_res, res.size());
    for (auto &r : res) max_len = std::max<int>(max_len, r.second.tokens.size());
  }
  res_dims[0] = max_res;
  res_dims[1] = max_len;
  if (max_res > max_results_cap || max_len > max_len_cap) return -1;
  for (size_t b = 0; b < results.size(); ++b) {
    for (size_t p = 0; p < results[b].size(); ++p) {
      const Output &o = results[b][p].second;
      size_t base = (b * max_results_cap + p) * static_cast<size_t>(max_len_cap);
      for (size_t t = 0; t < o.tokens.size(); ++t) {
        out_tokens[base + t] = o.tokens[t];
        out_timesteps[base + t] = o.timesteps[t];
      }
      out_scores[b * beam_stride + p] = static_cast<float>(results[b][p].first);
      out_lens[b * beam_stride + p] = static_cast<int>(o.tokens.size());
    }
  }
  return 1;
}

}  // extern "C"

// ---- scorer hooks for the product's host-side LM interface (include/ctcdecode_b200.h: ctcdec_scorer_hooks) -----
// These are what a maintainer of the reference would write in its own tree (INTEGRATION.md): the UNMODIFIED
// Scorer does the language-model work, the hook only turns a label-id prefix into the arguments it expects.
#include "lm/config.hh"
#include "lm/model.hh"

extern "C" {

// Scorer::get_log_cond_prob(Scorer::make_ngram(prefix)) for the prefix spelled by `labels` (scorer.cpp:74-93,163-194)
double ref_scorer_cond_from_labels(void *scorer, const int *labels, int n) {
  Scorer *s = static_cast<Scorer *>(scorer);
  std::vector<PathTrie> chain(static_cast<size_t>(n) + 1);  // chain[0] is the root (character == -1)
  for (int k = 0; k < n; ++k) {
    chain[k + 1].character = labels[k];
    chain[k + 1].parent = &chain[k];
  }
  return s->get_log_cond_prob(s->make_ngram(&chain[n]));
}

// Scorer::get_sent_log_prob(Scorer::split_labels(prefix))  (scorer.cpp:95-146)
double ref_scorer_sent_from_labels(void *scorer, const int *labels, int n) {
  Scorer *s = static_cast<Scorer *>(scorer);
  std::vector<int> v(labels, labels + n);
  return s->get_sent_log_prob(s->split_labels(v));
}

// Scorer::get_log_cond_prob(words) for one n-gram (scorer.cpp:74-93): what tests/golden/make_lm_tables.py records
double ref_scorer_cond_from_words(void *scorer, const char *const *words, int n) {
  return static_cast<Scorer *>(scorer)->get_log_cond_prob(std::vector<std::string>(words, words + n));
}

// The language model's vocabulary as KenLM enumerates it (what Scorer::load_lm collects, scorer.cpp:55-72),
// '\n'-separated into buf; returns the number of bytes needed.
size_t ref_lm_vocabulary(const char *lm_path, char *buf, size_t cap) {
  RetriveStrEnumerateVocab enumerate;
  lm::ngram::Config config;
  config.enumerate_vocab = &enumerate;
  lm::base::Model *m = lm::ngram::LoadVirtual(lm_path, config);
  delete m;
  std::string all;
  for (const std::string &w : enumerate.vocabulary) { all += w; all += '\n'; }
  if (buf && cap >= all.size() + 1) memcpy(buf, all.c_str(), all.size() + 1);
  return all.size() + 1;
}

}  // extern "C"
