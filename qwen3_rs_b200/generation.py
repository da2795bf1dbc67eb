"""Host-side generation loop on token ids, mirroring qwen3-inference/src/generation.rs.

The tokenizer / chat templates are out of scope (SURVEY.md §2 #8); callers pass token ids.
`generate` keeps the reference's quirk that prompt tokens except the last are never forwarded
(:26-28).  `generate_fast` is the drop-in speed-up: greedy decoding stays on the device
(q3_decode_greedy), only token ids cross PCIe."""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .sampler import Sampler


def generate_next_token(transformer, sampler: Sampler, token: int, pos: int) -> int:
    """generation.rs:153-162."""
    logits = transformer.forward(token, pos)  # forward() already returns a copy (logits.to_vec())
    return sampler.sample(logits)


def generate(transformer, sampler: Sampler, prompt_tokens: Sequence[int], max_new: Optional[int] = None,
             bos_token_id: int = -1, eos_token_id: int = -1) -> List[int]:
    """generation.rs:9-48.  Returns the sampled tokens (the terminating bos/eos is not included)."""
    if len(prompt_tokens) == 0:
        raise ValueError("Please provide a prompt")
    seq_len = transformer.get_config().seq_len
    pos, token, out = 0, int(prompt_tokens[0]), []
    while pos < seq_len and (max_new is None or len(out) < max_new):
        if pos < len(prompt_tokens) - 1:
            nxt = int(prompt_tokens[pos + 1])
        else:
            nxt = generate_next_token(transformer, sampler, token, pos)
            if nxt == bos_token_id or nxt == eos_token_id:
                break
            out.append(nxt)
        token = nxt
        pos += 1
    return out


def generate_fast(transformer, prompt_tokens: Sequence[int], max_new: int) -> List[int]:
    """Greedy `generate` with the decode loop resident on the GPU.  Same tokens as
    generate(..., Sampler(temperature=0)) without bos/eos termination."""
    if len(prompt_tokens) == 0:
        raise ValueError("Please provide a prompt")
    seq_len = transformer.get_config().seq_len
    pos0 = len(prompt_tokens) - 1
    n = max(0, min(max_new, seq_len - pos0))
    return transformer.decode_greedy(int(prompt_tokens[-1]), pos0, n)


def perplexity(transformer, tokens: Sequence[int], pos0: int = 0) -> Tuple[float, float]:
    """Perplexity of `tokens` placed at positions pos0.. -> (exp(-mean log p), sum log p) over the len(tokens) - 1 predictions
    tokens[1:], each conditioned on the tokens before it.  One q3_score pass; the KV cache then holds tokens[:-1]."""
    if len(tokens) < 2:
        raise ValueError("perplexity needs at least two tokens")
    seq_len = transformer.get_config().seq_len
    if pos0 < 0 or len(tokens) - 1 + pos0 > seq_len:
        raise ValueError(f"{len(tokens) - 1} scored positions from pos0 {pos0} exceed seq_len {seq_len}")
    lp, _ = transformer.score(list(tokens[:-1]), targets=list(tokens[1:]), pos0=pos0, want_argmax=False)
    total = float(np.sum(np.asarray(lp, np.float64)))
    return math.exp(-total / (len(tokens) - 1)), total


# ---------------------------------------------------------------------------------------------
# chat() on token ids (generation.rs:50-151).  The tokenizer and the prompt templates stay on the
# reference side: a "user turn" here is the already rendered + encoded prompt of that turn.
# ---------------------------------------------------------------------------------------------
class GenerationState:
    """generation.rs:236-257 (metrics omitted)."""

    def __init__(self, initial_token: int = 0):
        self.pos, self.token = 0, initial_token

    def reset(self, initial_token: int = 0):
        self.pos, self.token = 0, initial_token

    def advance(self, next_token: int):
        self.token, self.pos = next_token, self.pos + 1


def user_turn(transformer, sampler: Sampler, state: GenerationState, prompt_tokens: Sequence[int]) -> int:
    """handle_user_turn's token loop (generation.rs:116-122): one forward AND one sample per prompt token;
    only the last sample is used, the others merely advance the sampler's RNG.  Returns next_token."""
    seq_len = transformer.get_config().seq_len
    next_token = 0
    for token in prompt_tokens:
        if state.pos >= seq_len:
            break
        next_token = generate_next_token(transformer, sampler, int(token), state.pos)
        state.advance(int(token))
    return next_token


def user_turn_prefill(transformer, sampler: Sampler, state: GenerationState, prompt_tokens: Sequence[int]) -> int:
    """The drop-in for `user_turn`: the whole turn in ONE q3_prefill call (tensor-core GEMMs), sampling once
    from the last token's logits.  The reference draws one random number per discarded sample when
    temperature > 0 (sampler.rs:116-136: exactly one `random_f32` per `sample`, none for argmax), so the RNG
    is advanced by the same number of draws and a seeded run continues with the same stream."""
    seq_len = transformer.get_config().seq_len
    n = max(0, min(len(prompt_tokens), seq_len - state.pos))
    if n == 0:
        return 0
    logits = transformer.prefill([int(t) for t in prompt_tokens[:n]], state.pos)
    if sampler.temperature != 0.0:
        for _ in range(n - 1):
            sampler.random_u32()
    next_token = sampler.sample(logits)
    state.pos += n
    state.token = int(prompt_tokens[n - 1])
    return next_token


def chat(transformer, sampler: Sampler, turns, bos_token_id: int = -1, eos_token_id: int = -1,
         use_prefill: bool = True, max_new_per_turn: Optional[int] = None) -> List[List[int]]:
    """chat() (generation.rs:50-93, 128-151) over an iterable of encoded user turns; returns the assistant's
    tokens per turn.  As in the reference a full context window resets the position to 0 and hands the turn
    back to the user (:65-69); the KV cache is not cleared (attention only reads rows 0..=pos).
    `max_new_per_turn` is an addition (the reference generates until bos/eos or the window is full)."""
    seq_len = transformer.get_config().seq_len
    state = GenerationState(0)
    replies: List[List[int]] = []
    turns = iter(turns)
    is_user, next_token = True, 0
    while True:
        if state.pos >= seq_len:
            state.reset(0)
            is_user = True
        if is_user:
            prompt = next(turns, None)
            if prompt is None or len(prompt) == 0:
                break
            fn = user_turn_prefill if use_prefill else user_turn
            next_token = fn(transformer, sampler, state, prompt)
            replies.append([])
            is_user = False
        else:
            if next_token == bos_token_id or next_token == eos_token_id or \
                    (max_new_per_turn is not None and len(replies[-1]) >= max_new_per_turn):
                is_user = True
                continue
            replies[-1].append(next_token)
            next_token = generate_next_token(transformer, sampler, next_token, state.pos)
            state.advance(next_token)
    return replies
