// topk_check: qwen3::Transformer::score_topk through the C++ host header.
//   topk_check <checkpoint> <pos0> <k> <t0 t1 ...> -- <target0 target1 ...>
// Prints the top-k ids (one line, row-major), their log-probabilities as raw float bits (hex, one line), the target
// log-probabilities as raw bits (one line), the argmax tokens (one line), then the error code of a call with an out-of-range
// target (one line).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "qwen3_transformer.hpp"

static void print_bits(const std::vector<float> &v) {
    for (float x : v) {
        unsigned bits;
        std::memcpy(&bits, &x, 4);
        std::printf("%08x ", bits);
    }
    std::printf("\n");
}

int main(int argc, char **argv) {
    if (argc < 5) {
        std::fprintf(stderr, "usage: %s checkpoint pos0 k tokens... -- targets...\n", argv[0]);
        return 2;
    }
    const size_t pos0 = (size_t)std::atoi(argv[2]);
    const int k = std::atoi(argv[3]);
    std::vector<int> tokens, targets;
    bool after = false;
    for (int i = 4; i < argc; i++) {
        if (!std::strcmp(argv[i], "--")) after = true;
        else (after ? targets : tokens).push_back(std::atoi(argv[i]));
    }
    qwen3::Transformer t = qwen3::TransformerBuilder(argv[1]).build();
    const auto r = t.score_topk(tokens, k, targets, pos0);
    for (int id : r.ids) std::printf("%d ", id);
    std::printf("\n");
    print_bits(r.logprobs);
    print_bits(r.target_logprobs);
    for (int a : r.argmax) std::printf("%d ", a);
    std::printf("\n");
    std::vector<int> bad(targets);
    bad.back() = (int)t.get_config().vocab_size;
    try {
        t.score_topk(tokens, k, bad, pos0);
        std::printf("0\n");
    } catch (const qwen3::Error &e) {
        std::printf("%d\n", e.code());
    }
    return 0;
}
