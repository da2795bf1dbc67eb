// score_check: qwen3::Transformer::score through the C++ host header.
//   score_check <checkpoint> <pos0> <t0 t1 ...> -- <target0 target1 ...>
// Prints the log-probabilities as raw float bits (hex, one line), the argmax tokens (one line), then the error code of a
// call with an out-of-range target (one line).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "qwen3_transformer.hpp"

int main(int argc, char **argv) {
    if (argc < 4) {
        std::fprintf(stderr, "usage: %s checkpoint pos0 tokens... -- targets...\n", argv[0]);
        return 2;
    }
    const size_t pos0 = (size_t)std::atoi(argv[2]);
    std::vector<int> tokens, targets;
    bool after = false;
    for (int i = 3; i < argc; i++) {
        if (!std::strcmp(argv[i], "--")) after = true;
        else (after ? targets : tokens).push_back(std::atoi(argv[i]));
    }
    qwen3::Transformer t = qwen3::TransformerBuilder(argv[1]).build();
    auto res = t.score(tokens, targets, pos0);
    for (float v : res.first) {
        unsigned bits;
        std::memcpy(&bits, &v, 4);
        std::printf("%08x ", bits);
    }
    std::printf("\n");
    for (int a : res.second) std::printf("%d ", a);
    std::printf("\n");
    std::vector<int> bad(targets);
    bad.back() = (int)t.get_config().vocab_size;
    try {
        t.score(tokens, bad, pos0);
        std::printf("0\n");
    } catch (const qwen3::Error &e) {
        std::printf("%d\n", e.code());
    }
    return 0;
}
