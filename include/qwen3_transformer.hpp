// qwen3_transformer.hpp -- C++17 host-side mirror of the reference's interface for the quantized forward
// path, over the C ABI of libqwen3cuda (include/qwen3_cuda.h).  Header-only; link with -lqwen3cuda.
//
// The reference is Rust (toolchain absent from the build image), so the host layer a reference user
// programs against is restated here with the same names, argument meaning and error behaviour:
//
//   reference (qwen3-inference/src)                         here
//   ------------------------------------------------------  -----------------------------------------------
//   models/mod.rs:13-18   trait Transformer                  qwen3::Transformer::forward / get_config
//   models/mod.rs:40-74   TransformerBuilder                 qwen3::TransformerBuilder(path).with_ctx_length(..).build()
//   configuration.rs:18-30 ModelConfig                       qwen3::ModelConfig
//   sampler.rs            Sampler (xorshift64*, top-p)       qwen3::Sampler
//   layers.rs:495-506     softmax                            qwen3::softmax
//   generation.rs:9-48    generate                           qwen3::generate (token ids; tokenizer out of scope)
//   generation.rs:153-162 generate_next_token                qwen3::generate_next_token
//   generation.rs:50-151  chat (user / assistant turns)      qwen3::chat, user_turn, user_turn_prefill (one q3_prefill per turn)
//   tokenizer.rs          Tokenizer (byte-level BPE)         qwen3::Tokenizer (same results; vocabulary lookups hashed)
//   generation.rs:188-195 render_prompt                      qwen3::render_prompt
//
// Extensions of the drop-in (SURVEY section 8f): forward_argmax, decode_greedy, prefill, score, score_topk, forward_multi,
// decode_speculative.
//
// Errors: construction failures throw qwen3::Error (the reference returns anyhow::Error with the same
// message text); forward() with an out-of-range token / pos throws (the reference panics on the slice
// index).  There is no CPU fallback: without a CUDA device build() throws with code Q3_ECUDA.
//
// Bit-fidelity of Sampler/softmax with the reference needs IEEE semantics from the compiler building THIS
// header: no -ffast-math, no FMA contraction of `a*b+c` (gcc: -ffp-contract=off), as Rust never contracts.
#pragma once

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <optional>
#include <sstream>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "qwen3_cuda.h"

namespace qwen3 {

class Error : public std::runtime_error {
public:
    Error(int code, const std::string &what) : std::runtime_error(what), code_(code) {}
    int code() const { return code_; } // a Q3_E* value
private:
    int code_;
};

namespace detail {
inline void check(int rc) {
    if (rc != 0) {
        const char *m = q3_last_error();
        throw Error(rc, m ? m : "qwen3cuda error");
    }
}
// f32::total_cmp ordering key (sampler.rs:58, :87)
inline int32_t total_key(float f) {
    int32_t b;
    std::memcpy(&b, &f, 4);
    return b ^ (int32_t)(((uint32_t)(b >> 31)) >> 1);
}
} // namespace detail

// configuration.rs:18-30
struct ModelConfig {
    int dim = 0, hidden_dim = 0, n_layers = 0, n_heads = 0, n_kv_heads = 0, head_dim = 0, seq_len = 0, vocab_size = 0;
    int group_size = 0;
    bool shared_classifier = false;
    int architecture_id = 0;
};

// The `Transformers::Qwen3` variant (models/mod.rs:20-37) resident on one GPU.  Move-only; owns the handle.
class Transformer {
public:
    Transformer(const Transformer &) = delete;
    Transformer &operator=(const Transformer &) = delete;
    Transformer(Transformer &&o) noexcept : h_(o.h_), cfg_(o.cfg_), logits_(std::move(o.logits_)) { o.h_ = nullptr; }
    Transformer &operator=(Transformer &&o) noexcept {
        if (this != &o) {
            close();
            h_ = o.h_;
            cfg_ = o.cfg_;
            logits_ = std::move(o.logits_);
            o.h_ = nullptr;
        }
        return *this;
    }
    ~Transformer() { close(); }

    // Transformer::forward (models/mod.rs:15): logits of the next token, valid until the next call.
    const std::vector<float> &forward(size_t token, size_t pos) {
        detail::check(q3_forward(h_, (int)token, (int)pos, logits_.data()));
        return logits_;
    }
    const ModelConfig &get_config() const { return cfg_; }

    // ---- extensions ----
    size_t forward_argmax(size_t token, size_t pos) { // greedy token chosen on the device (sampler.rs:57-59 tie rule)
        int next = 0;
        detail::check(q3_forward_argmax(h_, (int)token, (int)pos, &next));
        return (size_t)next;
    }
    std::vector<int> decode_greedy(size_t first_token, size_t pos0, size_t n) { // whole greedy loop on the GPU
        std::vector<int> out(n ? n : 1);
        detail::check(q3_decode_greedy(h_, (int)first_token, (int)pos0, (int)n, out.data()));
        out.resize(n);
        return out;
    }
    // n prompt tokens at once (tensor-core GEMMs); cache and logits as after n sequential forwards
    const std::vector<float> &prefill(const std::vector<int> &tokens, size_t pos0) {
        detail::check(q3_prefill(h_, tokens.data(), (int)tokens.size(), (int)pos0, logits_.data()));
        return logits_;
    }
    // q3_score: tokens at positions pos0.. in one batched pass -> (log-probability of targets[i] after tokens[0..i], greedy
    // argmax there).  Empty targets: no log-probabilities (first vector empty).  Cache as after prefill(tokens, pos0).
    std::pair<std::vector<float>, std::vector<int>> score(const std::vector<int> &tokens, const std::vector<int> &targets, size_t pos0) {
        if (!targets.empty() && targets.size() != tokens.size()) throw std::invalid_argument("score: targets and tokens differ in length");
        std::vector<float> lp(targets.size());
        std::vector<int> am(tokens.size());
        detail::check(q3_score(h_, tokens.data(), (int)tokens.size(), (int)pos0, targets.empty() ? nullptr : targets.data(),
                               targets.empty() ? nullptr : lp.data(), am.data()));
        return {std::move(lp), std::move(am)};
    }
    // q3_score_topk: the k most likely tokens at every position, row-major [n][k] (most likely first, equal values with the
    // larger id first) and their log-probabilities; then score()'s two results (first empty without targets).
    struct TopK {
        std::vector<int> ids;
        std::vector<float> logprobs;
        std::vector<float> target_logprobs;
        std::vector<int> argmax;
    };
    TopK score_topk(const std::vector<int> &tokens, int k, const std::vector<int> &targets, size_t pos0) {
        if (!targets.empty() && targets.size() != tokens.size()) throw std::invalid_argument("score_topk: targets and tokens differ in length");
        if (k < 1 || k > Q3_TOPK_MAX) throw std::invalid_argument("score_topk: k outside 1 .. Q3_TOPK_MAX");
        TopK r;
        r.ids.resize(tokens.size() * (size_t)k);
        r.logprobs.resize(tokens.size() * (size_t)k);
        r.target_logprobs.resize(targets.size());
        r.argmax.resize(tokens.size());
        detail::check(q3_score_topk(h_, tokens.data(), (int)tokens.size(), (int)pos0, k, r.ids.data(), r.logprobs.data(),
                                    targets.empty() ? nullptr : targets.data(), targets.empty() ? nullptr : r.target_logprobs.data(),
                                    r.argmax.data()));
        return r;
    }
    // q3_forward_multi: tokens[i] at position pos0 + i (1 <= n <= Q3_MULTI_MAX) in one pass over the weights; the greedy token
    // after each prefix, and with want_logits the logits rows [n][vocab_size] (else empty).
    struct Multi {
        std::vector<int> argmax;
        std::vector<float> logits;
    };
    Multi forward_multi(const std::vector<int> &tokens, size_t pos0, bool want_logits = false) {
        if (tokens.empty() || tokens.size() > Q3_MULTI_MAX) throw std::invalid_argument("forward_multi: 1 .. Q3_MULTI_MAX tokens");
        Multi r;
        r.argmax.resize(tokens.size());
        if (want_logits) r.logits.resize(tokens.size() * (size_t)cfg_.vocab_size);
        detail::check(q3_forward_multi(h_, tokens.data(), (int)tokens.size(), (int)pos0, r.argmax.data(),
                                       want_logits ? r.logits.data() : nullptr));
        return r;
    }
    // q3_decode_speculative: n greedy tokens after first_token at pos0, k (1 .. Q3_MULTI_MAX - 1) drafted per round by `draft`;
    // the tokens of decode_greedy on the multi-kernel path.  Statistics of the rounds in the optional outputs.
    struct SpecStats {
        int rounds = 0, drafted = 0, accepted = 0;
    };
    std::vector<int> decode_speculative(Transformer &draft, int first_token, size_t pos0, size_t n, int k, SpecStats *stats = nullptr) {
        if (k < 1 || k > Q3_MULTI_MAX - 1) throw std::invalid_argument("decode_speculative: k outside 1 .. Q3_MULTI_MAX - 1");
        std::vector<int> out(n);
        SpecStats st;
        detail::check(q3_decode_speculative(h_, draft.h_, first_token, (int)pos0, (int)n, k, out.data(), &st.rounds, &st.drafted,
                                            &st.accepted));
        if (stats) *stats = st;
        return out;
    }
    void reset() { detail::check(q3_reset(h_)); } // zero the KV cache
    q3_handle *handle() { return h_; }

private:
    friend class TransformerBuilder;
    Transformer(q3_handle *h) : h_(h) {
        const q3_config *c = q3_get_config(h);
        cfg_.dim = c->dim;
        cfg_.hidden_dim = c->hidden_dim;
        cfg_.n_layers = c->n_layers;
        cfg_.n_heads = c->n_heads;
        cfg_.n_kv_heads = c->n_kv_heads;
        cfg_.head_dim = c->head_dim;
        cfg_.seq_len = c->seq_len;
        cfg_.vocab_size = c->vocab_size;
        cfg_.group_size = c->group_size;
        cfg_.shared_classifier = c->shared_classifier != 0;
        cfg_.architecture_id = c->architecture_id;
        logits_.resize((size_t)cfg_.vocab_size);
    }
    void close() {
        if (h_) q3_destroy(h_);
        h_ = nullptr;
    }
    q3_handle *h_ = nullptr;
    ModelConfig cfg_;
    std::vector<float> logits_;
};

// models/mod.rs:40-74
class TransformerBuilder {
public:
    explicit TransformerBuilder(std::string checkpoint_path) : path_(std::move(checkpoint_path)) {}
    TransformerBuilder &with_ctx_length(std::optional<int> ctx_length) { // None = the checkpoint's seq_len
        ctx_ = ctx_length;
        return *this;
    }
    TransformerBuilder &with_device(int device) { // addition: which GPU
        device_ = device;
        return *this;
    }
    Transformer build() const {
        q3_handle *h = nullptr;
        detail::check(q3_create(path_.c_str(), ctx_.value_or(0), device_, &h));
        return Transformer(h);
    }

private:
    std::string path_;
    std::optional<int> ctx_;
    int device_ = 0;
};

// layers.rs:495-506: subtract the maximum, exp, left-fold sum, multiply by 1/sum
inline void softmax(float *x, size_t n) {
    float mx = -INFINITY; // fold(NEG_INFINITY, f32::max): NaN-ignoring maximum
    for (size_t i = 0; i < n; i++) mx = std::fmax(mx, x[i]);
    float sum = 0.0f;
    for (size_t i = 0; i < n; i++) {
        x[i] = std::exp(x[i] - mx);
        sum += x[i];
    }
    const float inv = 1.0f / sum;
    for (size_t i = 0; i < n; i++) x[i] *= inv;
}

// sampler.rs
class Sampler {
public:
    float temperature, topp;
    uint64_t rng_state;

    Sampler(size_t vocab_size, float temperature_, float topp_, uint64_t rng_seed)
        : temperature(temperature_), topp(std::min(std::max(topp_, 0.0f), 1.0f)), rng_state(rng_seed), probindex_(vocab_size) {
        if (vocab_size == 0) throw std::invalid_argument("Vocab size must be positive");
        if (!(temperature_ >= 0.0f)) throw std::invalid_argument("Temperature must be non-negative");
        if (!(topp_ >= 0.0f && topp_ <= 1.0f)) throw std::invalid_argument("Top-p must be between 0.0 and 1.0");
    }

    uint32_t random_u32() { // :44-49 xorshift64*
        rng_state ^= rng_state >> 12;
        rng_state ^= rng_state << 25;
        rng_state ^= rng_state >> 27;
        return (uint32_t)((rng_state * 0x2545F4914F6CDD1DULL) >> 32);
    }
    float random_f32() { return (float)(random_u32() >> 8) / 16777216.0f; } // :52-54

    static size_t sample_argmax(const float *logits, size_t n) { // :57-59: max_by(total_cmp) keeps the LAST maximum
        size_t best = 0;
        for (size_t i = 1; i < n; i++)
            if (detail::total_key(logits[i]) >= detail::total_key(logits[best])) best = i;
        return best;
    }
    static size_t sample_mult(const float *p, size_t n, float coin) { // :62-71
        float cdf = 0.0f;
        for (size_t i = 0; i < n; i++) {
            cdf += p[i];
            if (coin < cdf) return i;
        }
        return n ? n - 1 : 0;
    }
    size_t sample_topp(const float *p, size_t n, float coin) { // :74-110
        const float cutoff = (1.0f - topp) / (float)std::max<size_t>(n ? n - 1 : 0, 1);
        size_t n0 = 0;
        for (size_t i = 0; i < n; i++)
            if (p[i] >= cutoff) probindex_[n0++] = {p[i], i};
        // the reference's sort_unstable_by leaves the order of equal probabilities unspecified; stable here
        std::stable_sort(probindex_.begin(), probindex_.begin() + (std::ptrdiff_t)n0,
                         [](const ProbIndex &a, const ProbIndex &b) { return detail::total_key(b.prob) < detail::total_key(a.prob); });
        float cumulative = 0.0f;
        size_t last = n0 ? n0 - 1 : 0;
        for (size_t i = 0; i < n0; i++) {
            cumulative += probindex_[i].prob;
            if (cumulative > topp) {
                last = i;
                break;
            }
        }
        const float r = coin * cumulative;
        float cdf = 0.0f;
        for (size_t i = 0; i <= last && i < n0; i++) {
            cdf += probindex_[i].prob;
            if (r < cdf) return probindex_[i].index;
        }
        return n0 ? probindex_[last].index : 0;
    }
    // :116-136 (modifies `logits` in place, as the reference does)
    size_t sample(float *logits, size_t n) {
        if (temperature == 0.0f) return sample_argmax(logits, n);
        for (size_t i = 0; i < n; i++) logits[i] /= temperature;
        softmax(logits, n);
        const float coin = random_f32();
        if (topp <= 0.0f || topp >= 1.0f) return sample_mult(logits, n, coin);
        return sample_topp(logits, n, coin);
    }
    size_t sample(std::vector<float> &logits) { return sample(logits.data(), logits.size()); }

private:
    struct ProbIndex {
        float prob;
        size_t index;
    };
    std::vector<ProbIndex> probindex_;
};

// The loops below are generic over the transformer type, like the reference's `T: Transformer` (generation.rs:9,50):
// anything with forward(token, pos) -> logits, get_config().seq_len and (for the prefill turn) prefill(tokens, pos0).

// generation.rs:153-162
template <class T>
size_t generate_next_token(T &t, Sampler &s, size_t token, size_t pos) {
    std::vector<float> logits = t.forward(token, pos); // logits.to_vec()
    return s.sample(logits);
}

// generation.rs:9-48 on token ids.  Prompt tokens except the last are never forwarded (:26-28); stops at
// bos/eos (not emitted), at seq_len, or after max_new tokens (addition; 0 = no cap).
template <class T>
std::vector<size_t> generate(T &t, Sampler &s, const std::vector<size_t> &prompt_tokens, size_t max_new = 0, long bos_token_id = -1,
                             long eos_token_id = -1) {
    if (prompt_tokens.empty()) throw std::invalid_argument("Please provide a prompt");
    const size_t seq_len = (size_t)t.get_config().seq_len;
    size_t pos = 0, token = prompt_tokens[0];
    std::vector<size_t> out;
    while (pos < seq_len && (max_new == 0 || out.size() < max_new)) {
        size_t next;
        if (pos + 1 < prompt_tokens.size()) {
            next = prompt_tokens[pos + 1];
        } else {
            next = generate_next_token(t, s, token, pos);
            if ((long)next == bos_token_id || (long)next == eos_token_id) break;
            out.push_back(next);
        }
        token = next;
        pos++;
    }
    return out;
}

// generation.rs:236-257 (metrics omitted)
struct GenerationState {
    size_t pos = 0, token = 0;
    void reset(size_t initial_token) {
        pos = 0;
        token = initial_token;
    }
    void advance(size_t next_token) {
        token = next_token;
        pos++;
    }
};

// handle_user_turn's token loop (generation.rs:116-122): one forward AND one sample per prompt token; only the last
// sample is used, the others merely advance the sampler's RNG.
template <class T>
size_t user_turn(T &t, Sampler &s, GenerationState &state, const std::vector<size_t> &prompt_tokens) {
    const size_t seq_len = (size_t)t.get_config().seq_len;
    size_t next_token = 0;
    for (size_t token : prompt_tokens) {
        if (state.pos >= seq_len) break;
        next_token = generate_next_token(t, s, token, state.pos);
        state.advance(token);
    }
    return next_token;
}

// The drop-in for user_turn: the whole turn in ONE prefill call, one sample from the last token's logits, and the RNG
// advanced by the draws the discarded samples would have made (Sampler::sample draws exactly one random_f32 per call
// when temperature > 0, none for argmax) - a seeded run continues with the same stream.
template <class T>
size_t user_turn_prefill(T &t, Sampler &s, GenerationState &state, const std::vector<size_t> &prompt_tokens) {
    const size_t seq_len = (size_t)t.get_config().seq_len;
    const size_t n = state.pos >= seq_len ? 0 : std::min(prompt_tokens.size(), seq_len - state.pos);
    if (n == 0) return 0;
    std::vector<int> ids(prompt_tokens.begin(), prompt_tokens.begin() + (std::ptrdiff_t)n);
    std::vector<float> logits = t.prefill(ids, state.pos);
    if (s.temperature != 0.0f)
        for (size_t i = 1; i < n; i++) s.random_u32();
    const size_t next_token = s.sample(logits);
    state.pos += n;
    state.token = prompt_tokens[n - 1];
    return next_token;
}

// chat() (generation.rs:50-93, 128-151) over already rendered + encoded user turns; returns the assistant's tokens per turn.
// A full context window resets the position and hands the turn back to the user (:65-69).  max_new_per_turn is an
// addition (0 = none: the reference generates until bos/eos or the window is full).
template <class T>
std::vector<std::vector<size_t>> chat(T &t, Sampler &s, const std::vector<std::vector<size_t>> &turns, long bos_token_id = -1,
                                      long eos_token_id = -1, bool use_prefill = true, size_t max_new_per_turn = 0) {
    const size_t seq_len = (size_t)t.get_config().seq_len;
    GenerationState state;
    std::vector<std::vector<size_t>> replies;
    size_t turn = 0, next_token = 0;
    bool is_user = true;
    while (true) {
        if (state.pos >= seq_len) {
            state.reset(0);
            is_user = true;
        }
        if (is_user) {
            if (turn >= turns.size() || turns[turn].empty()) break;
            next_token = use_prefill ? user_turn_prefill(t, s, state, turns[turn]) : user_turn(t, s, state, turns[turn]);
            turn++;
            replies.emplace_back();
            is_user = false;
        } else {
            if ((long)next_token == bos_token_id || (long)next_token == eos_token_id ||
                (max_new_per_turn != 0 && replies.back().size() >= max_new_per_turn)) {
                is_user = true;
                continue;
            }
            replies.back().push_back(next_token);
            next_token = generate_next_token(t, s, next_token, state.pos);
            state.advance(next_token);
        }
    }
    return replies;
}

// tokenizer.rs: byte-level BPE tokenizer read from `<checkpoint>.tokenizer` (+ the prompt templates next to it).
// Same token ids as the reference; its O(vocab) scans per lookup (`Iterator::position`, :145-151, :213-224) are
// replaced by a hash map that keeps the FIRST index of every byte string, which is what `position` returns.
class Tokenizer {
public:
    std::vector<std::string> vocab; // raw bytes, not necessarily valid UTF-8
    std::vector<float> merge_scores;
    size_t vocab_size = 0;
    uint32_t max_token_length = 0, bos_token_id = 0, eos_token_id = 0;
    std::string prompt_template, system_prompt_template;

    // Tokenizer::new (:40-100).  A file that ends early yields empty tokens with score 0, as in the reference.
    Tokenizer(const std::string &checkpoint_path, size_t vocab_size_, bool enable_thinking) : vocab_size(vocab_size_) {
        const std::string path = checkpoint_path + ".tokenizer";
        std::ifstream f(path, std::ios::binary);
        if (!f) throw std::runtime_error("cannot open " + path);
        if (!read_u32(f, max_token_length) || !read_u32(f, bos_token_id) || !read_u32(f, eos_token_id))
            throw std::runtime_error("short tokenizer header in " + path);
        vocab.reserve(vocab_size);
        merge_scores.reserve(vocab_size);
        for (size_t i = 0; i < vocab_size; i++) {
            float score;
            if (!f.read(reinterpret_cast<char *>(&score), 4)) {
                vocab.emplace_back();
                merge_scores.push_back(0.0f);
                continue;
            }
            merge_scores.push_back(score);
            uint32_t len;
            if (!read_u32(f, len)) {
                vocab.emplace_back();
                continue;
            }
            std::string bytes(len, '\0');
            if (len && !f.read(bytes.data(), len)) bytes.clear();
            vocab.push_back(std::move(bytes));
        }
        for (size_t i = 0; i < vocab.size(); i++) index_.emplace(vocab[i], i); // emplace keeps the first index
        prompt_template = load_prompt_template(checkpoint_path, false, enable_thinking);
        system_prompt_template = load_prompt_template(checkpoint_path, true, enable_thinking);
    }

    // :122-140: the token's bytes (the reference hands back the same bytes even when they are not valid UTF-8)
    std::string decode(size_t token) const { return token < vocab.size() ? vocab[token] : std::string(); }

    // :166-238
    std::vector<size_t> encode(const std::string &text) const {
        std::vector<std::string> chars = split_chars(text); // text.chars()
        std::vector<size_t> tokens;
        size_t i = 0;
        while (i < chars.size()) {
            bool found_special = false;
            if (chars[i] == "<") { // special tokens: "<...>" of at most max_token_length characters
                const size_t limit = std::min(chars.size(), i + (size_t)max_token_length);
                size_t end = 0;
                bool has_end = false;
                for (size_t j = i + 1; j < limit; j++) {
                    if (chars[j] == ">") {
                        end = j;
                        has_end = true;
                        break;
                    }
                }
                if (has_end) {
                    std::string special;
                    for (size_t j = i; j <= end; j++) special += chars[j];
                    auto it = index_.find(special);
                    if (it != index_.end()) {
                        tokens.push_back(it->second);
                        i = end + 1;
                        found_special = true;
                    }
                }
            }
            if (!found_special) {
                auto it = index_.find(chars[i]);
                if (it != index_.end()) tokens.push_back(it->second);
                else std::fprintf(stderr, "Warning: unknown character '%s' in input, skipping.\n", chars[i].c_str());
                i++;
            }
        }
        // merge the adjacent pair whose concatenation has the highest score until none is in the vocabulary;
        // strict `>`: among equal scores the leftmost pair wins
        while (true) {
            float best_score = -1e10f;
            size_t best_id = 0, best_idx = 0;
            bool found = false;
            for (size_t k = 0; k + 1 < tokens.size(); k++) {
                auto it = index_.find(vocab[tokens[k]] + vocab[tokens[k + 1]]);
                if (it != index_.end() && merge_scores[it->second] > best_score) {
                    best_score = merge_scores[it->second];
                    best_id = it->second;
                    best_idx = k;
                    found = true;
                }
            }
            if (!found) break;
            tokens[best_idx] = best_id;
            tokens.erase(tokens.begin() + (std::ptrdiff_t)best_idx + 1);
        }
        return tokens;
    }

private:
    static bool read_u32(std::ifstream &f, uint32_t &v) { return (bool)f.read(reinterpret_cast<char *>(&v), 4); } // little endian hosts
    // :103-119
    static std::string load_prompt_template(const std::string &checkpoint_path, bool with_system, bool enable_thinking) {
        const char *suffix = with_system ? (enable_thinking ? ".template.with-system-and-thinking" : ".template.with-system")
                                         : (enable_thinking ? ".template.with-thinking" : ".template");
        std::ifstream f(checkpoint_path + suffix, std::ios::binary);
        if (!f) {
            std::fprintf(stderr, "Warning: Could not load prompt template %s%s\n", checkpoint_path.c_str(), suffix);
            return std::string();
        }
        std::ostringstream ss;
        ss << f.rdbuf();
        return ss.str();
    }
    // Unicode scalar values of a UTF-8 string, each kept as its UTF-8 bytes (a stray byte counts as one character)
    static std::vector<std::string> split_chars(const std::string &s) {
        std::vector<std::string> out;
        for (size_t i = 0; i < s.size();) {
            const unsigned char c = (unsigned char)s[i];
            size_t n = c < 0x80 ? 1 : (c >> 5) == 0x6 ? 2 : (c >> 4) == 0xE ? 3 : (c >> 3) == 0x1E ? 4 : 1;
            if (i + n > s.size()) n = 1;
            for (size_t k = 1; k < n; k++)
                if (((unsigned char)s[i + k] >> 6) != 0x2) {
                    n = 1;
                    break;
                }
            out.emplace_back(s, i, n);
            i += n;
        }
        return out;
    }
    std::unordered_map<std::string, size_t> index_;
};

// generation.rs:188-195.  `str::replace` substitutes EVERY "%s" - in the system template both placeholders receive
// "{system}\n{user}" - which is what the reference does and therefore what this does.
inline std::string render_prompt(size_t pos, const std::optional<std::string> &system_prompt, const std::string &user_prompt,
                                 const Tokenizer &tokenizer) {
    auto replace_all = [](std::string tmpl, const std::string &with) {
        for (size_t at = tmpl.find("%s"); at != std::string::npos; at = tmpl.find("%s", at + with.size())) tmpl.replace(at, 2, with);
        return tmpl;
    };
    if (pos == 0 && system_prompt) return replace_all(tokenizer.system_prompt_template, *system_prompt + "\n" + user_prompt);
    return replace_all(tokenizer.prompt_template, user_prompt);
}

} // namespace qwen3
