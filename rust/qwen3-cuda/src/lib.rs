//! qwen3-cuda: `impl Transformer` over libqwen3cuda (B200 / sm_100a).
//!
//! NOT COMPILED in this repository (no Rust toolchain in the image); it is the reference-side binding
//! for include/qwen3_cuda.h.  It needs one line in qwen3-inference: `pub use
//! crate::configuration::ModelConfig;` (ModelConfig lives in a private module, lib.rs:5).
use anyhow::{bail, Result};
use qwen3_inference::{ModelConfig, Transformer};
use std::ffi::{c_char, c_float, c_int, CStr, CString};

#[repr(C)]
struct Q3Config {
    architecture_id: i32, dim: i32, hidden_dim: i32, n_layers: i32, n_heads: i32, n_kv_heads: i32,
    head_dim: i32, seq_len: i32, vocab_size: i32, group_size: i32, shared_classifier: i32,
}
#[repr(C)]
struct Q3Handle { _private: [u8; 0] }

extern "C" {
    fn q3_create(path: *const c_char, ctx_len: c_int, device: c_int, out: *mut *mut Q3Handle) -> c_int;
    fn q3_destroy(h: *mut Q3Handle);
    fn q3_get_config(h: *const Q3Handle) -> *const Q3Config;
    fn q3_forward(h: *mut Q3Handle, token: c_int, pos: c_int, logits_host: *mut c_float) -> c_int;
    fn q3_last_error() -> *const c_char;
    // extensions of the drop-in (no counterpart in the reference's trait)
    fn q3_forward_argmax(h: *mut Q3Handle, token: c_int, pos: c_int, next_token: *mut c_int) -> c_int;
    fn q3_decode_greedy(h: *mut Q3Handle, first_token: c_int, pos0: c_int, n: c_int, tokens_out: *mut c_int) -> c_int;
    fn q3_prefill(h: *mut Q3Handle, tokens: *const c_int, n: c_int, pos0: c_int, last_logits_host: *mut c_float) -> c_int;
    fn q3_score(h: *mut Q3Handle, tokens: *const c_int, n: c_int, pos0: c_int, targets: *const c_int, logprobs_out: *mut c_float,
                argmax_out: *mut c_int) -> c_int;
    fn q3_score_topk(h: *mut Q3Handle, tokens: *const c_int, n: c_int, pos0: c_int, k: c_int, topk_ids_out: *mut c_int,
                     topk_logprobs_out: *mut c_float, targets: *const c_int, logprobs_out: *mut c_float, argmax_out: *mut c_int)
                     -> c_int;
    fn q3_forward_multi(h: *mut Q3Handle, tokens: *const c_int, n: c_int, pos0: c_int, argmax_out: *mut c_int,
                        logits_host: *mut c_float) -> c_int;
    fn q3_decode_speculative(target: *mut Q3Handle, draft: *mut Q3Handle, first_token: c_int, pos0: c_int, n: c_int, k: c_int,
                             tokens_out: *mut c_int, rounds_out: *mut c_int, drafted_out: *mut c_int, accepted_out: *mut c_int)
                             -> c_int;
    fn q3_reset(h: *mut Q3Handle) -> c_int;
    fn q3_logits_host(h: *mut Q3Handle) -> *mut c_float;
}

fn last_error() -> String {
    unsafe { CStr::from_ptr(q3_last_error()).to_string_lossy().into_owned() }
}

/// Device-resident Qwen3 transformer; a drop-in for `Transformers::Qwen3` (models/mod.rs:20-37).
pub struct CudaTransformer {
    handle: *mut Q3Handle,
    config: ModelConfig,
    /// the handle's own page-locked logits buffer (q3_logits_host): `forward` DMA-s into it and lends it out, like the
    /// reference's `&self.buffers.logits` (models/qwen3.rs:78) -- no second host copy
    logits: *mut c_float,
}

impl CudaTransformer {
    /// `TransformerBuilder::new(path).with_ctx_length(ctx).build()` (models/mod.rs:46-73).
    pub fn build(checkpoint_path: &str, ctx_length: Option<usize>, device: i32) -> Result<Self> {
        let path = CString::new(checkpoint_path)?;
        let mut handle = std::ptr::null_mut();
        let rc = unsafe { q3_create(path.as_ptr(), ctx_length.unwrap_or(0) as c_int, device, &mut handle) };
        if rc != 0 {
            bail!("{}", last_error()); // same messages as configuration.rs:116-146 / models/mod.rs:57,71
        }
        let c = unsafe { &*q3_get_config(handle) };
        let config = ModelConfig {
            architecture_id: c.architecture_id as usize, dim: c.dim as usize, hidden_dim: c.hidden_dim as usize,
            n_layers: c.n_layers as usize, n_heads: c.n_heads as usize, n_kv_heads: c.n_kv_heads as usize,
            head_dim: c.head_dim as usize, seq_len: c.seq_len as usize, vocab_size: c.vocab_size as usize,
            group_size: c.group_size as usize, shared_classifier: c.shared_classifier != 0,
        };
        let logits = unsafe { q3_logits_host(handle) };
        Ok(Self { handle, config, logits })
    }

    /// Greedy token chosen on the device, same tie rule as `Sampler::sample_argmax` (sampler.rs:57-59).
    pub fn forward_argmax(&mut self, token: usize, pos: usize) -> usize {
        let mut next: c_int = 0;
        let rc = unsafe { q3_forward_argmax(self.handle, token as c_int, pos as c_int, &mut next) };
        if rc != 0 {
            panic!("{}", last_error());
        }
        next as usize
    }

    /// `n` greedy tokens with the loop resident on the GPU (what `generate` does at temperature 0).
    pub fn decode_greedy(&mut self, first_token: usize, pos0: usize, n: usize) -> Vec<usize> {
        let mut out = vec![0 as c_int; n.max(1)];
        let rc = unsafe { q3_decode_greedy(self.handle, first_token as c_int, pos0 as c_int, n as c_int, out.as_mut_ptr()) };
        if rc != 0 {
            panic!("{}", last_error());
        }
        out.truncate(n);
        out.into_iter().map(|t| t as usize).collect()
    }

    /// A whole prompt in one call (tensor-core GEMMs); cache and logits as after `tokens.len()` sequential forwards.
    /// For `handle_user_turn` (generation.rs:116-122): call this once, advance the sampler's RNG by
    /// `tokens.len() - 1` draws when temperature > 0, then sample once (see INTEGRATION.md).
    pub fn prefill(&mut self, tokens: &[usize], pos0: usize) -> &[f32] {
        let ids: Vec<c_int> = tokens.iter().map(|&t| t as c_int).collect();
        let rc = unsafe { q3_prefill(self.handle, ids.as_ptr(), ids.len() as c_int, pos0 as c_int, self.logits) };
        if rc != 0 {
            panic!("{}", last_error());
        }
        unsafe { std::slice::from_raw_parts(self.logits, self.config.vocab_size) }
    }

    /// Score `tokens` at positions pos0.. in one batched pass: (natural-log probability of `targets[i]` after tokens[..=i],
    /// greedy argmax there).  Perplexity of a text = exp(-mean) of `score(&text[..n - 1], &text[1..], 0).0`.
    pub fn score(&mut self, tokens: &[usize], targets: &[usize], pos0: usize) -> (Vec<f32>, Vec<usize>) {
        assert_eq!(tokens.len(), targets.len());
        let ids: Vec<c_int> = tokens.iter().map(|&t| t as c_int).collect();
        let tg: Vec<c_int> = targets.iter().map(|&t| t as c_int).collect();
        let mut lp = vec![0.0f32; ids.len()];
        let mut am = vec![0 as c_int; ids.len()];
        let rc = unsafe {
            q3_score(self.handle, ids.as_ptr(), ids.len() as c_int, pos0 as c_int, tg.as_ptr(), lp.as_mut_ptr(), am.as_mut_ptr())
        };
        if rc != 0 {
            panic!("{}", last_error());
        }
        (lp, am.into_iter().map(|a| a as usize).collect())
    }

    /// The `k` most likely tokens at every position of `tokens` (positions pos0..), in one batched pass: for each position
    /// `k` (token, natural-log probability) pairs, most likely first, equal values with the larger token id first
    /// (1 <= k <= min(64, vocab_size)).  The cache is left as by `score`.
    pub fn score_topk(&mut self, tokens: &[usize], k: usize, pos0: usize) -> Vec<Vec<(usize, f32)>> {
        let ids: Vec<c_int> = tokens.iter().map(|&t| t as c_int).collect();
        let mut top = vec![0 as c_int; ids.len() * k];
        let mut lps = vec![0.0f32; ids.len() * k];
        let rc = unsafe {
            q3_score_topk(self.handle, ids.as_ptr(), ids.len() as c_int, pos0 as c_int, k as c_int, top.as_mut_ptr(),
                          lps.as_mut_ptr(), std::ptr::null(), std::ptr::null_mut(), std::ptr::null_mut())
        };
        if rc != 0 {
            panic!("{}", last_error());
        }
        top.chunks(k.max(1)).zip(lps.chunks(k.max(1)))
            .map(|(t, l)| t.iter().zip(l).map(|(&i, &v)| (i as usize, v)).collect())
            .collect()
    }

    /// `tokens[i]` at position `pos0 + i` (1 ..= 8 tokens, `Q3_MULTI_MAX`) in one pass over the weights: the greedy token after
    /// each prefix, each bit-identical to a single-token step of the multi-kernel path.
    pub fn forward_multi(&mut self, tokens: &[usize], pos0: usize) -> Vec<usize> {
        let ids: Vec<c_int> = tokens.iter().map(|&t| t as c_int).collect();
        let mut am = vec![0 as c_int; ids.len()];
        let rc = unsafe {
            q3_forward_multi(self.handle, ids.as_ptr(), ids.len() as c_int, pos0 as c_int, am.as_mut_ptr(), std::ptr::null_mut())
        };
        if rc != 0 {
            panic!("{}", last_error());
        }
        am.into_iter().map(|t| t as usize).collect()
    }

    /// `n` greedy tokens after `first_token` at `pos0`, `k` (1 ..= 7) drafted per round by `draft` and verified in one pass:
    /// the tokens of `decode_greedy` on the multi-kernel path.  Returns the tokens and (rounds, drafted, accepted).
    pub fn decode_speculative(&mut self, draft: &mut CudaTransformer, first_token: usize, pos0: usize, n: usize, k: usize)
                              -> (Vec<usize>, (usize, usize, usize)) {
        let mut out = vec![0 as c_int; n.max(1)];
        let (mut r, mut d, mut a) = (0 as c_int, 0 as c_int, 0 as c_int);
        let rc = unsafe {
            q3_decode_speculative(self.handle, draft.handle, first_token as c_int, pos0 as c_int, n as c_int, k as c_int,
                                  out.as_mut_ptr(), &mut r, &mut d, &mut a)
        };
        if rc != 0 {
            panic!("{}", last_error());
        }
        out.truncate(n);
        (out.into_iter().map(|t| t as usize).collect(), (r as usize, d as usize, a as usize))
    }

    /// Zero the KV cache (a fresh `TransformerBlockBuffers`, qwen3.rs:439-440).
    pub fn reset(&mut self) {
        unsafe { q3_reset(self.handle) };
    }
}

impl Transformer for CudaTransformer {
    fn forward(&mut self, token: usize, pos: usize) -> &[f32] {
        let rc = unsafe { q3_forward(self.handle, token as c_int, pos as c_int, self.logits) };
        if rc != 0 {
            panic!("{}", last_error()); // the reference panics on out-of-range token/pos (slice index)
        }
        unsafe { std::slice::from_raw_parts(self.logits, self.config.vocab_size) }
    }
    fn get_config(&self) -> &ModelConfig {
        &self.config
    }
}

impl Drop for CudaTransformer {
    fn drop(&mut self) {
        unsafe { q3_destroy(self.handle) }
    }
}
// SAFETY: the handle is used through &mut self only (one caller at a time), like the reference.
unsafe impl Send for CudaTransformer {}
