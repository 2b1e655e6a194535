"""Text generation side path (reference scripts/train.py:577-654 `LlamaMultiModal.generate_batch`, called once per epoch at
train.py:1231-1241; the stage-1 script scripts/check_generation.py:131-222 drives the same call).

The reference monkey-patches the backbone's embedding layer and calls HF `generate(do_sample=True, temperature, top_k, top_p,
no_repeat_ngram_size=3, repetition_penalty=1.2)`.  Here the same sampler runs over the decoder kernels of libtcavp.so:
  * prefix = Q-Former image tokens (+ q_proj, + vision modality embedding) followed by the prompt embeddings (+ text modality
    embedding) — `Engine.prefix_embeds`, the assembly of train.py:585-598;
  * every step evaluates the decoder stack over the sequence so far (`Engine.llm_forward`: tcgen05 GEMMs, tcgen05 / flash attention)
    and the vocabulary logits of the LAST position with one M = B GEMM against lm_head;
  * logits processors in HF's order: repetition penalty -> no-repeat-ngram -> temperature -> top-k -> top-p -> multinomial draw.
Decoding uses a KV cache (SURVEY.md §8 f4; Llama- and GPT-2-arch backbones): the prefix is evaluated once (`Engine.llm_forward(kv_out=...)` keeps every
layer's rotated keys / values), then every new token is one `Engine.llm_decode_step` — a one-row pass through the same kernels whose
query attends over the cached positions.  `kv_cache=False` recomputes the sequence so far at every step, which is also what the cached
path is tested against.  The sampled tokens depend on torch's RNG, the logits do not.

`seed=<int>` selects the device loop instead (KV cache only): after the eager prefill, one decode iteration — embed the sampled tokens,
`Engine.llm_decode_step_device`, lm_head, `tcavp_sample_next` — is captured in a CUDA graph and replayed once per new token.  The
position lives in device memory and the sampler advances it, so the loop makes no blocking host read; sampling is a pure function of
(seed, row, step) (counter hash, include/tcavp.h) instead of torch's RNG, so a run is reproducible from its seed.  Same processors, same
greedy tokens, different random draws than the default path.

Deviation from the reference, on purpose: the reference's patched embedding returns `fused_embeds[:, :len(ids)]` on the first call, i.e.
it silently drops the last 16 prompt positions and hands HF an attention mask that is 16 longer than the input (train.py:604-611,
627-632).  This implementation generates after the FULL prefix (image tokens + whole prompt), which is what the surrounding code intends."""
import torch

from . import ops

MAX_DECODE_LOOPS = 4     # captured decode loops kept per engine (least recently used dropped first)
CAPTURES = 0             # decode-loop captures in this process


@torch.no_grad()
def next_token_logits(engine, embeds, mask=None):
    """embeds (B, L, H) in the activation dtype -> fp32 logits (B, V) of the token that follows position L - 1."""
    B, L, H = embeds.shape
    if mask is None:
        mask = torch.ones(B, L, dtype=torch.int32, device=embeds.device)
    fh = engine.llm_forward(embeds.clone(), mask, B, L)                    # (B * L, H), post final norm (= hidden_states[-1])
    last = fh.view(B, L, H)[:, L - 1].contiguous()
    head = engine.lm_head()
    logits = torch.empty(B, head.shape[0], dtype=torch.float32, device=embeds.device)
    return ops.gemm(last, head, logits)


def process_logits(logits, seq, temperature, top_k, top_p, repetition_penalty, no_repeat_ngram_size):
    """HF's LogitsProcessorList of `generate(do_sample=True, ...)` for one step; `seq` (B, T) = token ids so far (prompt + generated)."""
    B, V = logits.shape
    if repetition_penalty and repetition_penalty != 1.0 and seq.shape[1] > 0:      # RepetitionPenaltyLogitsProcessor
        score = torch.gather(logits, 1, seq)
        score = torch.where(score < 0, score * repetition_penalty, score / repetition_penalty)
        logits = logits.scatter(1, seq, score)
    n = int(no_repeat_ngram_size or 0)
    if n > 0 and seq.shape[1] + 1 >= n:                                             # NoRepeatNGramLogitsProcessor
        for b in range(B):
            ids = seq[b].tolist()
            prefix = tuple(ids[len(ids) - (n - 1):]) if n > 1 else ()
            banned = [ids[i + n - 1] for i in range(len(ids) - n + 1) if tuple(ids[i:i + n - 1]) == prefix]
            if banned:
                logits[b, torch.tensor(banned, device=logits.device)] = float("-inf")
    if temperature and temperature != 1.0:                                          # TemperatureLogitsWarper
        logits = logits / temperature
    if top_k and 0 < top_k < V:                                                     # TopKLogitsWarper
        kth = torch.topk(logits, top_k, dim=-1).values[:, -1:]
        logits = logits.masked_fill(logits < kth, float("-inf"))
    if top_p is not None and 0.0 < top_p < 1.0:                                     # TopPLogitsWarper (keeps at least one token)
        srt, idx = torch.sort(logits, descending=False, dim=-1)
        cum = srt.softmax(dim=-1).cumsum(dim=-1)
        remove = cum <= (1.0 - top_p)
        remove[:, -1] = False
        logits = logits.masked_fill(torch.zeros_like(remove).scatter(1, idx, remove), float("-inf"))
    return logits


@torch.no_grad()
def generate_ids(model, vision_embs, prompt_ids, max_new_tokens=128, temperature=0.9, top_k=40, top_p=0.9, do_sample=True,
                 repetition_penalty=1.2, no_repeat_ngram_size=3, eos_token_id=None, pad_token_id=None, generator=None, kv_cache=True, seed=None):
    """-> (B, prompt + new) token ids: the prompt followed by the generated tokens (rows that hit `eos_token_id` are padded).
    `seed` (int): the device loop (module docstring): sampling reproducible from the seed, no host synchronisation per token; needs
    kv_cache=True and no `generator`."""
    if seed is not None:
        if isinstance(seed, bool) or not isinstance(seed, int):
            raise ValueError(f"seed must be an int (got {type(seed).__name__})")
        if not kv_cache:
            raise ValueError("seed needs kv_cache=True: the device loop decodes from the KV cache")
        if generator is not None:
            raise ValueError("seed and generator are exclusive: with a seed the draws come from the counter hash, not from a torch generator")
        return _generate_device(model, vision_embs, prompt_ids, int(max_new_tokens), seed, dict(
            do_sample=bool(do_sample), temperature=float(temperature) if do_sample else 1.0, top_k=int(top_k or 0) if do_sample else 0,
            top_p=(None if top_p is None else float(top_p)) if do_sample else None, repetition_penalty=float(repetition_penalty or 1.0),
            no_repeat_ngram_size=int(no_repeat_ngram_size or 0), eos_token_id=eos_token_id, pad_token_id=pad_token_id))
    eng = model.engine()
    dev = eng.dev
    ids = prompt_ids.to(device=dev, dtype=torch.int64)
    B = ids.shape[0]
    prefix = eng.prefix_embeds(vision_embs, ids)                           # (B, Q + Lp, H)
    P, H = prefix.shape[1], prefix.shape[2]
    seq = ids.clone()
    new_embeds = []
    done = torch.zeros(B, dtype=torch.bool, device=dev)
    pad = eos_token_id if pad_token_id is None else pad_token_id
    use_cache = bool(kv_cache) and int(max_new_tokens) > 0
    caches, head, logits = [], eng.lm_head(), None
    if use_cache:      # prefill: one pass over the prefix, keys / values of every layer kept
        ones = torch.ones(B, P, dtype=torch.int32, device=dev)
        fh = eng.llm_forward(prefix.clone(), ones, B, P, kv_out=(caches, P + int(max_new_tokens)))
        logits = ops.gemm(fh.view(B, P, H)[:, P - 1].contiguous(), head, torch.empty(B, head.shape[0], dtype=torch.float32, device=dev))
    for step in range(int(max_new_tokens)):
        if not use_cache:
            embeds = prefix if not new_embeds else torch.cat([prefix] + new_embeds, dim=1)
            logits = next_token_logits(eng, embeds)
        logits = process_logits(logits, seq, temperature if do_sample else 1.0, top_k if do_sample else 0, top_p if do_sample else None,
                                repetition_penalty, no_repeat_ngram_size)
        if do_sample:
            nxt = torch.multinomial(logits.softmax(dim=-1), 1, generator=generator)[:, 0]
        else:
            nxt = logits.argmax(dim=-1)
        if eos_token_id is not None:
            nxt = torch.where(done, torch.full_like(nxt, pad if pad is not None else 0), nxt)
            done = done | (nxt == eos_token_id)
        seq = torch.cat([seq, nxt[:, None]], dim=1)
        emb = eng.token_embeds(nxt[:, None])                               # plain embedding rows (no modality vector): train.py:609-611
        if eos_token_id is not None and bool(done.all()):
            break
        if use_cache:
            if step + 1 < int(max_new_tokens):
                h = eng.llm_decode_step(emb.view(B, H), caches, P + step)
                logits = ops.gemm(h, head, torch.empty(B, head.shape[0], dtype=torch.float32, device=dev))
        else:
            new_embeds.append(emb)
    return seq


def generate_batch(model, vision_embs, prompt_ids, tokenizer, max_new_tokens=128, temperature=0.9, top_k=40, top_p=0.9, device="cuda", seed=None):
    """Drop-in for `LlamaMultiModal.generate_batch` (train.py:577-654): list of decoded strings, cut after the reference's end marker.
    `seed`: the device loop of generate_ids."""
    was_training = model.training
    model.eval()
    try:
        out = generate_ids(model, vision_embs, prompt_ids, max_new_tokens=max_new_tokens, temperature=temperature, top_k=top_k, top_p=top_p,
                           eos_token_id=getattr(tokenizer, "eos_token_id", None), pad_token_id=getattr(tokenizer, "pad_token_id", None),
                           seed=seed)
    finally:
        model.train(was_training)
    texts = []
    marker = "No right-following vehicle."                                 # train.py:648-652
    for row in out:
        text = tokenizer.decode(row, skip_special_tokens=True)
        if marker in text:
            text = text[: text.index(marker) + len(marker)]
        texts.append(text)
    return texts


class DecodeLoop:
    """The static buffers of one (B, prefix length, prompt length, new tokens, sampling parameters) on one engine and the CUDA graph of
    one decode iteration over them: embed the tokens just sampled, `Engine.llm_decode_step_device` at position P - 1 + step, lm_head,
    tcavp_sample_next (which appends the next token and advances the step).  `run` fills the caches with the eager prefill, samples the
    first token and replays the graph for the others."""

    def __init__(self, eng, B, P, Lp, n_new, sp):
        global CAPTURES
        m, dev = eng.llm, eng.dev
        self.eng, self.B, self.P, self.Lp, self.n_new, self.sp = eng, B, P, Lp, n_new, sp
        self.cap = P + n_new
        width = 2 * (m["nh"] if m.get("arch") == "gpt2" else m["nkv"]) * m["dh"]
        self.caches = [torch.zeros(B, self.cap, width, dtype=eng.act, device=dev) for _ in m["layers"]]
        self.head = eng.lm_head()
        V = self.head.shape[0]
        self.logits = torch.zeros(B, V, dtype=torch.float32, device=dev)
        self.work = torch.empty(B, V, dtype=torch.float32, device=dev)
        self.hist = torch.zeros(B, Lp + n_new, dtype=torch.int64, device=dev)
        self.tokens = torch.zeros(B, dtype=torch.int64, device=dev)
        self.state = torch.zeros(3, dtype=torch.int32, device=dev)       # step, arrival counter, all-done step
        self.done = torch.zeros(B, dtype=torch.int32, device=dev)
        self.seed = torch.zeros(2, dtype=torch.int32, device=dev)
        self.ws = eng.decode_workspace(B, self.cap)
        self.flag = torch.zeros(1, dtype=torch.int32, pin_memory=True)
        self.graph = None
        if n_new > 1:
            # one eager iteration on a side stream (RoPE table, allocator warm-up; the buffers it scribbles on are reset by run()), then capture
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self.iteration()
            torch.cuda.current_stream().wait_stream(s)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.iteration()
            CAPTURES += 1

    def sample(self):
        ops.sample_next(self.logits, self.work, self.hist, self.state, self.done, self.tokens, hist_offset=self.Lp, seed=self.seed, **self.sp)

    def iteration(self):
        h = self.eng.llm_decode_step_device(self.tokens, self.caches, self.state, self.P - 1, self.ws)
        ops.gemm(h, self.head, self.logits)
        self.sample()

    def run(self, prefix, ids, seed):
        """-> (B, Lp + generated) ids, trimmed as the eager loop trims them (at the first step after which every row is done)."""
        eng, B, P, H = self.eng, self.B, self.P, prefix.shape[2]
        s = int(seed) & 0xFFFFFFFFFFFFFFFF
        words = [w - (1 << 32) if w >= (1 << 31) else w for w in (s & 0xFFFFFFFF, s >> 32)]
        self.seed[0].fill_(words[0])
        self.seed[1].fill_(words[1])
        self.state.zero_()
        self.done.zero_()
        self.hist[:, :self.Lp].copy_(ids)
        ones = torch.ones(B, P, dtype=torch.int32, device=eng.dev)
        fh = eng.llm_forward(prefix.clone(), ones, B, P, kv_out=(self.caches, self.cap))
        ops.gemm(fh.view(B, P, H)[:, P - 1].contiguous(), self.head, self.logits)
        self.sample()
        _device_loop(self, self.n_new - 1)
        n = int(self.state[2]) or self.n_new          # after the loop: the one host read of the call
        return self.hist[:, :self.Lp + n].clone()


def _device_loop(loop, n):
    """Replays the decode iteration up to n times.  When an EOS id is set, the all-done step is polled without blocking (a copy to pinned
    memory behind an event that is only queried) and the loop stops once it is seen; the replays it may run past that point only append pad."""
    poll = loop.sp["eos_token_id"] is not None
    pending = None
    for _ in range(n):
        if pending is not None and pending.query():
            if int(loop.flag[0]):
                break
            pending = None
        loop.graph.replay()
        if poll and pending is None:
            loop.flag.copy_(loop.state[2:3], non_blocking=True)
            pending = torch.cuda.Event()
            pending.record()


@torch.no_grad()
def _generate_device(model, vision_embs, prompt_ids, max_new_tokens, seed, sp):
    eng = model.engine()
    ids = prompt_ids.to(device=eng.dev, dtype=torch.int64)
    B, Lp = ids.shape
    prefix = eng.prefix_embeds(vision_embs, ids)
    P = prefix.shape[1]
    if max_new_tokens <= 0:
        return ids.clone()
    m = eng.llm
    if m.get("arch") == "gpt2" and P + max_new_tokens - 1 > m["wpe"].shape[0]:
        raise ops._lib.TcavpError(f"decode position {P + max_new_tokens - 2} is past the cache capacity {P + max_new_tokens} / n_positions "
                                  f"{m['wpe'].shape[0]}")
    loops = eng.__dict__.setdefault("_decode_loops", {})
    key = (B, P, Lp, max_new_tokens, tuple(sorted(sp.items())))
    loop = loops.pop(key, None)
    if loop is None:
        loop = DecodeLoop(eng, B, P, Lp, max_new_tokens, sp)
        while len(loops) >= MAX_DECODE_LOOPS:
            loops.pop(next(iter(loops)))          # dicts keep insertion order: the first key is the least recently used
    loops[key] = loop                             # (re-)inserted last = most recently used
    return loop.run(prefix, ids, seed)
