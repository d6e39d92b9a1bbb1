#!/usr/bin/env python
"""bench.py — decode tokens/s + p50 TTFT of the Server-CRD inference hot path (BASELINE.json metric).

A "step" is one synthetic request batch through the hot path: B prompts of 512 token ids
(randint(0,V), seed 1234+i; SURVEY.md §8d) -> prefill -> 127 further greedy decode steps (128 new tokens).
  value  = decode tokens/s, whole job, device-timed (CUDA events on the engine stream), inputs resident in HBM
           (the decode loop feeds tokens back on the device);
  e2e    = the same metric through the public C-ABI call with HOST buffers (ssb_prefill / ssb_decode take host
           token ids and return host token ids; host<->device copies inside the timed region, wall clock);
  ttft   = p50 wall time of ssb_prefill (host ids in -> first token id on the host).
Weights are seeded synthetic values at the real shapes (no checkpoints exist offline).
Inputs are larger than L2 (13.2 GB of weights stream per decode step vs 126 MB L2) so no L2 flush is needed.

The headline line is BASELINE configs[1] (Llama-2-7B bf16, batch 1).  The same line carries the other BASELINE configs
as sub-objects so that the driver's runs record them:
  N = 1 : batch32 (config 2, batch 32), llama2_13b_q4_gguf_b32 (config 3: a synthetic Q4_0 GGUF file written to local
          disk, dequant-on-load -> bf16, batch 32), falcon_40b (config 4 at TP1), llama2_70b (config 5's TP1 anchor),
          opt_125m_cpu_container (config 1: the reference's CPU container restated, one greedy request), cpu_baseline;
  N > 1 : batch32, tp_parity (TP-N vs TP1 logits on the workload's own weights, ids equal across ranks, tiny model vs
          the CPU oracle), llama2_70b (TP-N, with the TP1 anchor re-measured on rank 0), falcon_40b (N = 2, 4).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference] [--no-extras] [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PROMPT_LEN, NEW_TOKENS = 512, 128
TTFT_SAMPLES = 20  # SURVEY.md 8d: p50 TTFT over >= 20 requests

WORKLOADS = {
    # "tiny" exists for the CPU contract test of the reference arm (tests/test_bench_contract.py), not for benchmarking
    "tiny": dict(model_type="llama", hidden_size=256, intermediate_size=688, num_hidden_layers=8, num_attention_heads=2,
                 num_key_value_heads=2, vocab_size=512, max_position_embeddings=512, rms_norm_eps=1e-5, rope_theta=10000.0,
                 tie_word_embeddings=False, torch_dtype="bfloat16"),
    "llama2-7b": dict(model_type="llama", hidden_size=4096, intermediate_size=11008, num_hidden_layers=32,
                      num_attention_heads=32, num_key_value_heads=32, vocab_size=32000, max_position_embeddings=4096,
                      rms_norm_eps=1e-5, rope_theta=10000.0, tie_word_embeddings=False, torch_dtype="bfloat16"),
    "llama2-13b": dict(model_type="llama", hidden_size=5120, intermediate_size=13824, num_hidden_layers=40,
                       num_attention_heads=40, num_key_value_heads=40, vocab_size=32000, max_position_embeddings=4096,
                       rms_norm_eps=1e-5, rope_theta=10000.0, tie_word_embeddings=False, torch_dtype="bfloat16"),
    # BASELINE config 4 (examples/falcon-40b): new_decoder_architecture, 128 query / 8 KV heads of 64, GELU MLP 4h, parallel block
    "falcon-40b": dict(model_type="falcon", hidden_size=8192, num_hidden_layers=60, num_attention_heads=128, num_kv_heads=8,
                       vocab_size=65024, layer_norm_epsilon=1e-5, new_decoder_architecture=True, parallel_attn=True, bias=False,
                       alibi=False, multi_query=True, rope_theta=10000.0, max_position_embeddings=2048,
                       tie_word_embeddings=False, torch_dtype="bfloat16"),
    "tiny-falcon": dict(model_type="falcon", hidden_size=256, num_hidden_layers=6, num_attention_heads=4, num_kv_heads=2,
                        vocab_size=512, layer_norm_epsilon=1e-5, new_decoder_architecture=True, parallel_attn=True, bias=False,
                        alibi=False, multi_query=True, rope_theta=10000.0, max_position_embeddings=512,
                        tie_word_embeddings=False, torch_dtype="bfloat16"),
    "llama2-70b": dict(model_type="llama", hidden_size=8192, intermediate_size=28672, num_hidden_layers=80,
                       num_attention_heads=64, num_key_value_heads=8, vocab_size=32000, max_position_embeddings=4096,
                       rms_norm_eps=1e-5, rope_theta=10000.0, tie_word_embeddings=False, torch_dtype="bfloat16"),
    # BASELINE config 1 (examples/facebook-opt-125m): real OPT-125m shapes, CPU reference container only
    "opt-125m": dict(model_type="opt", architectures=["OPTForCausalLM"], hidden_size=768, ffn_dim=3072, num_hidden_layers=12,
                     num_attention_heads=12, vocab_size=50272, max_position_embeddings=2048, word_embed_proj_dim=768,
                     do_layer_norm_before=True, activation_function="relu", pad_token_id=1, bos_token_id=2, eos_token_id=2,
                     torch_dtype="float16"),
}
# tensor-parallel parity model: every sharded dimension divides by 8 (16 heads / 8 KV heads of 128, inter 2816 = 8 * 352)
TP_TINY = dict(model_type="llama", hidden_size=2048, intermediate_size=2816, num_hidden_layers=3, num_attention_heads=16,
               num_key_value_heads=8, vocab_size=1008, max_position_embeddings=512, rms_norm_eps=1e-5, rope_theta=10000.0,
               tie_word_embeddings=False, torch_dtype="bfloat16")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def synthetic_prompts(vocab, batch, plen):
    import torch

    rows = []
    for i in range(batch):
        g = torch.Generator().manual_seed(1234 + i)
        rows.append(torch.randint(0, vocab, (plen,), generator=g).tolist())
    return rows


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ===================================================================================================== CPU reference arm
def _host_threads():
    # cores this process may actually use (cgroup / affinity), capped: torch's CPU GEMV collapses when oversubscribed
    # (measured on the GPU box in round 1: 128 threads -> 0.04 tok/s, 25 s per token)
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return max(1, min(avail, 32))


def _hf_cpu_model(cfg, dtype):
    """The reference's CPU serving library (HF transformers, the library the Basaran image wraps) at cfg's FULL depth, eager
    attention, random weights.  Parameters are filled by tiling one small uniform block (memcpy speed; values are finite
    and of the real scale, which is all a timing needs — a 27 GB torch.uniform_ alone would take a minute)."""
    import torch

    fam = cfg.get("model_type")
    if fam == "falcon":
        from transformers import FalconConfig as Config, FalconForCausalLM as Model
        from transformers.models.falcon.modeling_falcon import FalconRotaryEmbedding as Rotary
    elif fam == "opt":
        from transformers import OPTConfig as Config, OPTForCausalLM as Model
        Rotary = None
    else:
        from transformers import LlamaConfig as Config, LlamaForCausalLM as Model
        from transformers.models.llama.modeling_llama import LlamaRotaryEmbedding as Rotary
    keys = {k: v for k, v in cfg.items() if k not in ("model_type", "torch_dtype", "rope_theta", "architectures")}
    if Rotary is not None:
        keys["rope_parameters"] = {"rope_type": "default", "rope_theta": cfg.get("rope_theta", 10000.0)}
    hcfg = Config(**keys, attn_implementation="eager")
    with torch.device("meta"):
        m = Model(hcfg)
    n_params = sum(p.numel() for p in m.parameters())
    need = n_params * torch.finfo(dtype).bits // 8
    try:
        import psutil

        avail = psutil.virtual_memory().available
    except Exception:
        avail = None
    if avail is not None and need > 0.8 * avail:
        raise MemoryError(f"n/a (host RAM): {need / 1e9:.0f} GB of {str(dtype).split('.')[-1]} weights, {avail / 1e9:.0f} GB available")
    m = m.to_empty(device="cpu").to(dtype)
    g = torch.Generator().manual_seed(0)
    block = torch.empty(1 << 22, dtype=dtype).uniform_(-0.0346, 0.0346, generator=g)  # std 0.02, HF's initializer_range
    with torch.no_grad():
        for name, p in m.named_parameters():
            if p.dim() >= 2:
                flat = p.view(-1)
                for o in range(0, flat.numel(), block.numel()):
                    n = min(block.numel(), flat.numel() - o)
                    flat[o:o + n].copy_(block[:n])
            else:
                p.fill_(0.0 if name.endswith("bias") else 1.0)
        for name, b in m.named_buffers():
            if b.dtype.is_floating_point and "inv_freq" not in name:
                b.zero_()
    if Rotary is not None:
        (m.transformer if fam == "falcon" else m.model).rotary_emb = Rotary(hcfg)  # to_empty() dropped the inv_freq buffer
    return m.eval(), n_params


def hf_cpu_measure(cfg, steps, warmup, prompt_len, tok_cap, batch=1, dtype="float32"):
    """ONE full-depth request on the host cores — no layer extrapolation: prefill of the workload's own seeded prompt
    (TTFT), then (warmup + steps) decode steps of T greedy tokens each, continuing the same sequence; T is chosen after
    timing one token so that a step is ~6 s at most, and (warmup + steps) * T never exceeds the workload's 127 decode
    tokens.  fp32: HF's default dtype on CPU (bf16 GEMV has no fast path on these hosts: 38 s per token measured in round 1)."""
    import torch

    threads = _host_threads()
    torch.set_num_threads(threads)
    dt = getattr(torch, dtype)
    t0 = time.time()
    m, n_params = _hf_cpu_model(cfg, dt)
    build_s = time.time() - t0
    ids = torch.tensor(synthetic_prompts(cfg["vocab_size"], batch, prompt_len))
    with torch.no_grad():
        t1 = time.time()
        out = m(ids, use_cache=True)
        nxt = out.logits[:, -1].float().argmax(-1)
        ttft = time.time() - t1
        past = out.past_key_values

        def tokens(n):
            nonlocal past, nxt
            t = time.time()
            for _ in range(n):
                o = m(nxt[:, None], past_key_values=past, use_cache=True)
                past = o.past_key_values
                nxt = o.logits[:, -1].float().argmax(-1)
            return time.time() - t

        t_tok = tokens(1)  # also the warm-up of the decode path
        n_steps = max(1, steps) + max(0, warmup)
        T = max(1, min(tok_cap, int(6.0 / max(t_tok, 1e-6)), max(1, (NEW_TOKENS - 2) // n_steps)))
        for _ in range(max(0, warmup)):
            tokens(T)
        step_s = [tokens(T) for _ in range(max(1, steps))]
    del m, past
    # the host is shared (128 cores, other tenants): a burst in one step moved the MEAN by 30 % between driver runs, so the
    # reported rate is tokens per step over the MEDIAN step time
    tok_s = batch * T / statistics.median(step_s)
    return {"decode_tok_s": tok_s, "ttft_s": ttft, "threads": threads, "cores": os.cpu_count(), "build_s": build_s, "dtype": dtype,
            "tokens_per_step": T, "step_ms": [s * 1e3 for s in step_s], "n_params": n_params,
            "sample": f"one full-depth ({cfg.get('num_hidden_layers')} layers, {n_params / 1e9:.2f} G params) request: {batch}x {prompt_len}-token seeded prompt "
                      f"prefilled once, then {len(step_s)} timed steps (+{max(0, warmup)} warm-up) of {T} greedy decode tokens each on the growing context (rate from the median step); "
                      f"HF transformers {dtype} eager (HF's CPU default dtype), {threads} host threads"}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU serving path (HF transformers) timed on the host cores.  Rank 0 only."""
    if rank != 0:
        return
    cfg = WORKLOADS[args.workload]
    base = {"impl": "reference", "metric": "decode_tokens_per_sec", "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    try:
        r = hf_cpu_measure(cfg, args.steps, args.warmup, args.ref_prompt_len, args.ref_new_tokens, batch=args.batch)
    except MemoryError as ex:
        print(json.dumps(dict(base, value=None, unavailable=str(ex), config={"workload": f"{args.workload} decode, batch {args.batch}, CPU reference path"},
                              cpu_baseline={"value": None, "unit": "tokens/s", "cores": _host_threads(), "kind": "reference", "sample": str(ex)})), flush=True)
        return
    v = r["decode_tok_s"]
    line = dict(base, value=v, ms_per_step=statistics.median(r["step_ms"]), ms_per_step_mean=statistics.mean(r["step_ms"]), tokens_per_step=r["tokens_per_step"],
                config={"workload": f"{args.workload} decode, batch {args.batch}, {args.ref_prompt_len}-token prompt, CPU reference path", "sample": r["sample"]},
                ttft_ms_p50=r["ttft_s"] * 1e3, model_build_s=r["build_s"],
                cpu_baseline={"value": v, "unit": "tokens/s", "cores": r["threads"], "kind": "reference", "sample": r["sample"]},
                e2e={"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    print(json.dumps(line), flush=True)


def opt_125m_container_line():
    """BASELINE config 1: examples/facebook-opt-125m through the reference's CPU container restated (oracle/ref_server.py =
    HF transformers behind `GET /` + `POST /v1/completions`, test/system.sh:73-78), real OPT-125m shapes, random weights,
    ONE greedy request of 16 prompt ids -> 32 tokens over HTTP.  Plumbing, no GPU."""
    import urllib.request

    from oracle import ref_server

    d = tempfile.mkdtemp(prefix="ssb_opt_")
    with open(os.path.join(d, "config.json"), "w") as f:
        json.dump(WORKLOADS["opt-125m"], f)
    import torch

    torch.set_num_threads(_host_threads())
    t0 = time.time()
    srv = ref_server.serve(d, 0, "float32")
    port = srv.server_address[1]
    threading.Thread(target=srv.serve_forever, daemon=True).start()

    def req(path, data=None):
        r = urllib.request.Request(f"http://127.0.0.1:{port}{path}", data=json.dumps(data).encode() if data is not None else None,
                                   headers={"Content-Type": "application/json"})
        with urllib.request.urlopen(r, timeout=120) as f_:
            return f_.status, json.loads(f_.read())

    try:
        for _ in range(1200):
            try:
                if req("/")[0] == 200:
                    break
            except Exception:
                pass
            time.sleep(0.1)
        ready_s = time.time() - t0
        prompt = synthetic_prompts(50272, 1, 16)[0]
        w0 = time.time()
        st, r = req("/v1/completions", {"prompt": prompt, "max_tokens": 32})
        wall = time.time() - w0
        return {"status": st, "value": r["decode_tokens_per_sec"], "unit": "tokens/s", "ttft_ms": r["ttft_ms"], "request_wall_s": wall,
                "pod_ready_s": ready_s, "completion_tokens": r["usage"]["completion_tokens"], "threads": _host_threads(),
                "config": "facebook/opt-125m shapes (h768 L12 H12 ffn3072 V50272), fp32, HF transformers CPU container restated, 16-token prompt + 32 greedy tokens, 1 request"}
    finally:
        srv.shutdown()


# ===================================================================================================== B200 arm
class Ctx:
    def __init__(self, args):
        import torch

        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.torch = torch
        self.dist = None
        self.peak_gbs, self.peak_src = load_peaks()
        self.extra_params = json.loads(args.engine_params) if args.engine_params else {}

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def all_ok(self, ok: bool) -> bool:
        """True only if every rank says ok (collective)."""
        if self.world == 1:
            return ok
        t = self.torch.tensor([1 if ok else 0], device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item())

    def max_over_ranks(self, v: float) -> float:
        if self.world == 1:
            return v
        from substratus_b200 import tp

        return tp.max_over_ranks(v)


def make_engine(cx: Ctx, model_dir: str, params: dict, tp_world=None):
    """Create (and, under TP, connect) an engine on this rank.  Collective when tp_world > 1.  Returns (engine, load_s)."""
    from substratus_b200 import Engine

    w = cx.world if tp_world is None else tp_world
    p = dict(params, device=cx.local_rank, tp_size=w, tp_rank=cx.rank if w > 1 else 0)
    t0 = time.time()
    eng, err = None, None
    try:
        eng = Engine(model_dir, p)
    except Exception as ex:
        err = ex
    if w > 1:
        if not cx.all_ok(err is None):
            if eng is not None:
                eng.close()
            raise RuntimeError(f"engine creation failed on some rank: {err!r}")
        from substratus_b200 import tp

        tp.connect(eng)  # all-gather the CUDA-IPC handles of the exchange buffers; the allreduce then runs over NVLink
    elif err is not None:
        raise err
    return eng, time.time() - t0


def config_dir(cfg: dict) -> str:
    tmp = tempfile.mkdtemp(prefix="ssb_bench_")
    with open(os.path.join(tmp, "config.json"), "w") as f:
        json.dump(cfg, f)
    return tmp


def measure(cx: Ctx, eng, vocab, B, steps, warmup, ttft_samples=TTFT_SAMPLES, collective=True):
    """K timed request batches of size B after W warm-ups; device times are MAX over ranks (collective=False: this rank alone)."""
    prompts = synthetic_prompts(vocab, B, PROMPT_LEN)
    info = eng.info
    mx = cx.max_over_ranks if collective else (lambda v: v)

    outputs = {}

    def one_request():
        sids = [eng.seq_create() for _ in range(B)]
        w0 = time.perf_counter()
        first, _ = eng.prefill(sids, prompts)  # host ids in (H2D inside), first token id back on the host
        w1 = time.perf_counter()
        pre_ms = eng.timing().prefill_ms
        rest, _ = eng.decode(sids, first, NEW_TOKENS - 1)  # 127 device-resident steps, ids back on the host (D2H inside)
        w2 = time.perf_counter()
        dec_ms = eng.timing().decode_ms
        for s in sids:
            eng.seq_free(s)
        outputs.update(prefill_tokens=first, decode_tokens=rest)  # the ids the caller receives; the top-up prefills below keep these
        return dict(ttft_wall_ms=(w1 - w0) * 1e3, prefill_dev_ms=pre_ms, decode_dev_ms=dec_ms,
                    decode_wall_ms=(w2 - w1) * 1e3, total_wall_ms=(w2 - w0) * 1e3)

    for _ in range(warmup):
        one_request()
    eng.timing_reset()
    sampler = ClockSampler(cx.local_rank)
    sampler.start()
    if collective:
        cx.barrier()
    else:
        cx.torch.cuda.synchronize()
    t0 = time.perf_counter()
    recs = [one_request() for _ in range(steps)]
    if collective:
        cx.barrier()
    else:
        cx.torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    wall = mx(wall)
    for r in recs:
        for k in r:
            r[k] = mx(r[k])
    tm = eng.timing()
    # SURVEY.md 8d quotes p50 TTFT over >= 20 requests after the warm-ups: top the K timed requests up with prefill-only
    # requests.  They run after the timed region and after the counters were read, so value / e2e / launches / bytes
    # are those of the K steps alone.
    ttfts = [r["ttft_wall_ms"] for r in recs]
    pre_devs = [r["prefill_dev_ms"] for r in recs]
    for _ in range(max(0, ttft_samples - steps)):
        sids = [eng.seq_create() for _ in range(B)]
        w0 = time.perf_counter()
        eng.prefill(sids, prompts)
        t_ms = (time.perf_counter() - w0) * 1e3
        d_ms = eng.timing().prefill_ms
        for sid in sids:
            eng.seq_free(sid)
        ttfts.append(mx(t_ms))
        pre_devs.append(mx(d_ms))
    ctx_mean = PROMPT_LEN + (NEW_TOKENS - 1) / 2.0 + 0.5
    ntok = B * (NEW_TOKENS - 1)
    dec_dev_s = sum(r["decode_dev_ms"] for r in recs) / 1e3
    dec_wall_s = sum(r["decode_wall_ms"] for r in recs) / 1e3
    bytes_step = info.weight_bytes_per_step + B * ctx_mean * info.kv_bytes_per_token
    step_ms = dec_dev_s * 1e3 / (steps * (NEW_TOKENS - 1))
    step_gbs = bytes_step / (step_ms * 1e-3) / 1e9
    return dict(value=steps * ntok / dec_dev_s, e2e=steps * ntok / dec_wall_s, wall=wall, clocks=clocks, tm=tm,
                ttft_ms_p50=statistics.median(ttfts), prefill_device_ms_p50=statistics.median(pre_devs), ttft_samples=len(ttfts),
                request_tok_s=steps * B * NEW_TOKENS / (sum(r["total_wall_ms"] for r in recs) / 1e3),
                step_ms=step_ms, bytes_step=bytes_step, step_gbs=step_gbs, ctx_mean=ctx_mean, outputs=outputs)


def compact(cx: Ctx, m, B, load_s, eng, what):
    """Sub-object form of one measurement."""
    return {"config": what, "value": m["value"], "unit": "tokens/s", "e2e": m["e2e"], "batch": B, "ttft_ms_p50": m["ttft_ms_p50"],
            "decode_ms_per_step": m["step_ms"], "bytes_per_step_per_gpu": m["bytes_step"], "hbm_gbs_per_gpu": m["step_gbs"],
            "hbm_roofline_frac": m["step_gbs"] / cx.peak_gbs, "roofline_tok_s": B * cx.peak_gbs * 1e9 / m["bytes_step"],
            "load_s": load_s, "hbm_gb": eng.info.hbm_bytes_allocated / 1e9, "clocks": m["clocks"]}


def sub_bench(cx: Ctx, workload, B, steps, warmup, what, tp_world=None, extra=None, ttft_samples=6):
    """One more BASELINE config inside the same run: synthetic weights on the device, its own engine."""
    cfg = WORKLOADS[workload]
    params = {"weights": "synthetic", "seed": 0, "max_batch": max(B, 4), "max_seq_len": PROMPT_LEN + NEW_TOKENS + 16,
              "use_pdl": cx.args.pdl, "use_graph": cx.args.graph}
    params.update(cx.extra_params)
    params.update(extra or {})
    collective = (cx.world if tp_world is None else tp_world) > 1
    eng, load_s = make_engine(cx, config_dir(cfg), params, tp_world)
    try:
        m = measure(cx, eng, cfg["vocab_size"], B, steps, warmup, ttft_samples=ttft_samples, collective=collective)
        return compact(cx, m, B, load_s, eng, what)
    finally:
        eng.close()


def write_q4_0_gguf(path, cfg, seed=0):
    """A synthetic Q4_0 GGUF `model.bin` at cfg's shapes (examples/llama2-13b-chat-gguf/base-model.yaml:8-9 stores exactly one
    such file): llama.cpp's container and tensor names, every weight matrix as Q4_0 blocks (fp16 scale of the real
    magnitude + 32 random 4-bit values), norms as F32.  Blocks come from one random pool read at tensor-specific offsets —
    the engine's reader, H2D copies and dequant kernel do the same work as for a trained file.  Returns the file size."""
    import numpy as np
    from gguf import GGMLQuantizationType as T
    from gguf import GGUFWriter

    rng = np.random.default_rng(seed)
    h, nh, nkv = cfg["hidden_size"], cfg["num_attention_heads"], cfg["num_key_value_heads"]
    inter, v, L = cfg["intermediate_size"], cfg["vocab_size"], cfg["num_hidden_layers"]
    w = GGUFWriter(path, "llama")
    w.add_context_length(cfg["max_position_embeddings"])
    w.add_embedding_length(h)
    w.add_block_count(L)
    w.add_feed_forward_length(inter)
    w.add_head_count(nh)
    w.add_head_count_kv(nkv)
    w.add_layer_norm_rms_eps(cfg["rms_norm_eps"])
    w.add_rope_freq_base(cfg["rope_theta"])
    d = h // nh
    biggest = max(v * h, inter * h) // 32
    n_pool = biggest + (1 << 16)
    pool = rng.integers(0, 256, size=(n_pool, 18), dtype=np.uint8)
    pool[:, 0:2] = (0.0346 / 8.0 * (0.5 + rng.random(n_pool, dtype=np.float32))).astype(np.float16).view(np.uint8).reshape(n_pool, 2)
    k = [0]

    def q4(name, rows, cols):
        nb = rows * cols // 32
        off = (k[0] * 7919) % (1 << 16)
        k[0] += 1
        w.add_tensor(name, pool[off:off + nb].reshape(rows, cols // 32 * 18), raw_dtype=T.Q4_0)

    q4("token_embd.weight", v, h)
    for l in range(L):
        p = f"blk.{l}."
        q4(p + "attn_q.weight", nh * d, h)
        q4(p + "attn_k.weight", nkv * d, h)
        q4(p + "attn_v.weight", nkv * d, h)
        q4(p + "attn_output.weight", h, nh * d)
        q4(p + "ffn_gate.weight", inter, h)
        q4(p + "ffn_up.weight", inter, h)
        q4(p + "ffn_down.weight", h, inter)
        w.add_tensor(p + "attn_norm.weight", np.ones(h, dtype=np.float32))
        w.add_tensor(p + "ffn_norm.weight", np.ones(h, dtype=np.float32))
    w.add_tensor("output_norm.weight", np.ones(h, dtype=np.float32))
    q4("output.weight", v, h)
    w.write_header_to_file()
    w.write_kv_data_to_file()
    w.write_tensors_to_file()
    w.close()
    return os.path.getsize(path)


def gguf_bench(cx: Ctx, steps, warmup):
    """BASELINE config 3: Llama-2-13B from a Q4_0 GGUF file on local disk, dequant-on-load -> bf16, decode batch 32."""
    cfg = WORKLOADS["llama2-13b"]
    d = tempfile.mkdtemp(prefix="ssb_gguf_", dir="/dev/shm" if os.path.isdir("/dev/shm") and _shm_has_room() else None)
    path = os.path.join(d, "model.bin")
    t0 = time.time()
    size = write_q4_0_gguf(path, cfg)
    write_s = time.time() - t0
    try:
        eng, load_s = make_engine(cx, d, {"max_batch": 32, "max_seq_len": PROMPT_LEN + NEW_TOKENS + 16, "use_pdl": cx.args.pdl,
                                          "use_graph": cx.args.graph}, tp_world=1)
        try:
            m = measure(cx, eng, cfg["vocab_size"], 32, steps, warmup, ttft_samples=4, collective=False)
            out = compact(cx, m, 32, load_s, eng, "llama2-13b Q4_0 GGUF file -> dequant-on-load -> bf16, decode batch 32, 512+128, 1xB200")
            out.update({"gguf_file_gb": size / 1e9, "gguf_write_s": write_s, "gguf_dir": os.path.dirname(d),
                        "load_s_note": "ssb_engine_create: GGUF parse + H2D of the raw blocks + dequant kernel + row permutation, file in the page cache"})
            return out
        finally:
            eng.close()
    finally:
        try:
            os.remove(path)
            os.rmdir(d)
        except OSError:
            pass


def _shm_has_room():
    try:
        st = os.statvfs("/dev/shm")
        return st.f_bavail * st.f_frsize > 12 * (1 << 30)
    except OSError:
        return False


def tp_parity(cx: Ctx):
    """Tensor-parallel correctness carried by the bench line (the driver's GPU test box has one GPU): (1) a small GQA model
    at TP-N against the CPU oracle (same criterion as tests/test_parity_gpu.py, ids equal on every rank); (2) the
    workload's own weights: TP-N logits against a TP1 engine on rank 0 for a fixed 64-token prompt + 4 decode steps."""
    import numpy as np
    torch, dist = cx.torch, cx.dist
    out = {}

    def gather_tokens(toks):
        t = torch.tensor(np.asarray(toks, dtype=np.int64), device="cuda")
        all_t = [torch.empty_like(t) for _ in range(cx.world)]
        dist.all_gather(all_t, t)
        return bool(all(torch.equal(all_t[0], x) for x in all_t))

    def rel(a, b):
        a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
        return float(np.abs(a - b).max() / np.abs(b).max())

    base = {"weights": "synthetic", "max_batch": 4, "max_seq_len": 160}
    base.update(cx.extra_params)
    # (1) tiny model vs oracle
    g = torch.Generator().manual_seed(5)
    prompts = [torch.randint(0, TP_TINY["vocab_size"], (n,), generator=g).tolist() for n in (19, 40)]
    eng, _ = make_engine(cx, config_dir(TP_TINY), dict(base, seed=17))
    try:
        toks, lg = eng.generate(prompts, 6, want_logits=True)
    finally:
        eng.close()
    out["tiny_ids_equal_across_ranks"] = gather_tokens(toks)
    if cx.rank == 0:
        from oracle import llama_ref, synth

        sd = synth.llama_state_dict(TP_TINY, 17)
        lgt = np.transpose(lg, (1, 0, 2))
        errs = {}
        for name, dt in (("f32", torch.float32), ("bf16", torch.bfloat16)):
            ref = llama_ref.LlamaRef(TP_TINY, sd, dt)
            rows = []
            for p, t in zip(prompts, toks):
                ref.reset()
                rows.append(ref.forward(torch.tensor([list(p) + [int(x) for x in t[:-1]]]))[0, len(p) - 1:].float().numpy())
            errs[name] = np.stack(rows)
        eg = np.array([[rel(lgt[i, s], errs["f32"][i, s]) for s in range(6)] for i in range(2)])
        ec = np.array([[rel(errs["bf16"][i, s], errs["f32"][i, s]) for s in range(6)] for i in range(2)])
        ids_ok = all(int(errs["f32"][i, s].argmax()) == int(toks[i, s]) or
                     float(errs["f32"][i, s].max() - errs["f32"][i, s, toks[i, s]]) < 4 * float(np.abs(errs["bf16"] - errs["f32"]).max())
                     for i in range(2) for s in range(6))
        out.update({"tiny_model": "llama h2048 H16 KV8 I2816 L3 V1008, synthetic seed 17, 2 prompts x 6 tokens",
                    "tiny_err_gpu_mean_vs_fp32_oracle": float(eg.mean()), "tiny_err_cpu_bf16_mean_vs_fp32_oracle": float(ec.mean()),
                    "tiny_err_gpu_max": float(eg.max()), "tiny_err_cpu_bf16_max": float(ec.max()),
                    "tiny_pass": bool(eg.mean() <= ec.mean() + 1e-3 and eg.max() <= 1.5 * ec.max() + 1e-3),
                    "tiny_greedy_ids_match_fp32_oracle_or_tie": bool(ids_ok)})
    # (2) the workload's own weights, TP-N vs TP1
    wl = cx.args.workload
    cfg = WORKLOADS[wl]
    prompt = synthetic_prompts(cfg["vocab_size"], 1, 64)
    eng, _ = make_engine(cx, config_dir(cfg), dict(base, seed=0))
    try:
        toksN, lgN = eng.generate(prompt, 5, want_logits=True)
    finally:
        eng.close()
    out["workload_ids_equal_across_ranks"] = gather_tokens(toksN)
    cx.barrier()
    if cx.rank == 0:
        try:
            e1, _ = make_engine(cx, config_dir(cfg), dict(base, seed=0), tp_world=1)
            try:
                sid = e1.seq_create()
                first, l0 = e1.prefill([sid], prompt, want_logits=True)
                forced = [int(x) for x in toksN[0]]
                # teacher-force the TP-N ids so that every step compares logits for the same context
                lg1 = [l0[0]]
                for s in range(4):
                    _, l = e1.decode([sid], [forced[s]], 1, want_logits=True)
                    lg1.append(l[0, 0])
                e1.seq_free(sid)
            finally:
                e1.close()
            errs = [rel(lgN[s, 0], lg1[s]) for s in range(5)]
            out.update({"workload": f"{wl}, 64-token seeded prompt + 4 decode steps, TP{cx.world} vs TP1 (teacher-forced with the TP{cx.world} ids)",
                        "workload_logits_rel_err_vs_tp1": errs, "workload_logits_rel_err_vs_tp1_max": max(errs),
                        "workload_ids_equal_tp1": bool(all(int(np.argmax(lg1[s])) == forced[s] for s in range(5))),
                        # two bf16 evaluations of the full-depth model with different fp32 summation orders (TP-N sums N partials per
                        # row-parallel projection): the CPU bf16 oracle itself sits 7e-2 from the fp32 truth at 32 layers
                        # (tests/test_fullwidth_gpu.py::test_full_depth_7b_vs_fp32_oracle), so "same function" = well inside 2 x that
                        "workload_rel_err_bound": 1e-1, "workload_pass": bool(max(errs) < 1e-1)})
        except Exception as ex:
            out["workload_error"] = repr(ex)
    cx.barrier()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--workload", default="llama2-7b", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batch32", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sub-objects for the other BASELINE configs")
    ap.add_argument("--extras", default="", help="comma list restricting the sub-objects: gguf13b,falcon40b,llama70b,opt125m,tp_parity")
    ap.add_argument("--ref-prompt-len", type=int, default=PROMPT_LEN)
    ap.add_argument("--ref-new-tokens", type=int, default=8, help="reference arm: decode tokens per timed step (upper bound)")
    ap.add_argument("--pdl", type=int, default=1)
    ap.add_argument("--graph", type=int, default=1)
    ap.add_argument("--engine-params", default="", help="JSON object merged into the engine's params.json (experiments, e.g. "
                    "'{\"tp_mega\": 1}'); echoed in config.engine_params so an overridden run is never mistaken for the default")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the token ids the last timed request returned (prefill_tokens [B], "
                         "decode_tokens [B, 127]) as float32 DIR/<name>.npy; inputs are seeded, so two builds compare id for id")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the serving path has no CPU fallback (use --impl reference for the CPU arm)")
    cx = Ctx(args)
    torch.cuda.set_device(cx.local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", cx.local_rank))
        cx.dist = dist
    cfg = WORKLOADS[args.workload]
    peak_gbs, peak_src = cx.peak_gbs, cx.peak_src
    extra_params = cx.extra_params
    params = {"weights": "synthetic", "seed": 0, "max_batch": max(args.batch, 32), "max_seq_len": PROMPT_LEN + NEW_TOKENS + 16,
              "use_pdl": args.pdl, "use_graph": args.graph}
    params.update(extra_params)
    eng, t_load = make_engine(cx, config_dir(cfg), params)
    info = eng.info

    B = args.batch
    m = measure(cx, eng, cfg["vocab_size"], B, args.steps, args.warmup)
    if args.dump_outputs and cx.rank == 0:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in m["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.asarray(a, dtype=np.float32))  # ids < 2^24: exact
    launches = int(m["tm"].kernel_launches)
    h2d, d2h = m["tm"].h2d_bytes // args.steps, m["tm"].d2h_bytes // args.steps

    # Dominant kernel.  At batch <= 4 the whole decode step IS one kernel (decode_mega_kernel; under tensor parallelism too,
    # with the allreduce inside it): its achieved bandwidth is the step's algorithmic bytes over its CUDA-event duration.
    # Otherwise the dominant kernel is the gate/up projection (44% of the weight bytes), timed live with ssb_bench_kernel.
    kern = {}
    for k in ("gate_up", "qkv", "down", "o", "lm_head", "attn"):
        ms, by = eng.bench_kernel(k, rows=B, ctx=int(m["ctx_mean"]), iters=64)
        kern[k] = {"ms": ms, "bytes": by, "gbs": by / (ms * 1e-3) / 1e9}
    tp_mega_on = extra_params.get("tp_mega", TP_MEGA_DEFAULT) if world > 1 else 1
    mega = B <= 4 and cfg.get("model_type") != "falcon" and bool(tp_mega_on) and extra_params.get("use_mega", 1) != 0
    if mega:
        roofline = {"bound": "hbm", "kernel": "decode_mega_kernel (persistent single-kernel decode step: all projections, attention, pick"
                                              + (", in-kernel NVLink allreduce)" if world > 1 else ")"),
                    "achieved": m["step_gbs"], "peak": peak_gbs, "unit": "GB/s", "frac": m["step_gbs"] / peak_gbs,
                    "traffic": MEGA_TRAFFIC_BYTES.get((args.workload, B, world)), "algorithmic_bytes_per_launch": m["bytes_step"],
                    "ms_per_launch": m["step_ms"]}
    else:
        dom = kern["gate_up"]
        roofline = {"bound": "hbm", "kernel": "gate/up projection (proj_rows_kernel for <= 4 rows, tc_gemm_sk_kernel tcgen05 stream-K above)",
                    "achieved": dom["gbs"], "peak": peak_gbs, "unit": "GB/s", "frac": dom["gbs"] / peak_gbs, "traffic": None,
                    "algorithmic_bytes_per_launch": dom["bytes"], "ms_per_launch": dom["ms"]}
    roofline.update({"peak_source": peak_src, "per_kernel_class_gbs": {k: round(v["gbs"], 1) for k, v in kern.items()},
                     "decode_step": {"bytes": m["bytes_step"], "ms": m["step_ms"], "achieved": m["step_gbs"],
                                     "frac": m["step_gbs"] / peak_gbs, "roofline_tok_s": B * peak_gbs * 1e9 / m["bytes_step"]}})

    line = {
        "metric": "decode_tokens_per_sec", "value": m["value"], "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": m["wall"] * 1e3 / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.workload} bf16 decode, batch {B}, {PROMPT_LEN}-token prompt + {NEW_TOKENS} new tokens, {world}xB200",
                   "batch": B, "prompt_len": PROMPT_LEN, "new_tokens": NEW_TOKENS, "parallelism": f"tp{world}",
                   "allreduce": ("inside the persistent decode kernel: 16-byte {value, epoch} pushes into every rank's receive slots over NVLink peer "
                                 "memory (CUDA IPC), receiver polls the slot; prefill: one-shot pull allreduce kernel") if world > 1 and mega else
                                ("one-shot pull allreduce kernel over NVLink peer memory (CUDA IPC)" if world > 1 else "none"),
                   "l2": "inputs larger than L2 (weights streamed per decode step >> 126 MB)", "pdl": args.pdl, "graph": args.graph},
        "ttft_ms_p50": m["ttft_ms_p50"], "ttft_samples": m["ttft_samples"], "prefill_device_ms_p50": m["prefill_device_ms_p50"],
        "decode_ms_per_token": m["step_ms"],
        "e2e": {"value": m["e2e"], "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "request_tokens_per_sec": m["request_tok_s"]},
        "gpu_launches": launches, "clocks": m["clocks"], "roofline": roofline, "load_s": t_load,
        "hbm_gb": info.hbm_bytes_allocated / 1e9,
    }
    if world > 1:
        n_ar = 2 * cfg["num_hidden_layers"] if cfg.get("model_type") != "falcon" else cfg["num_hidden_layers"]
        ideal_ms = m["bytes_step"] / (peak_gbs * 1e9) * 1e3
        line["tp"] = {"allreduces_per_token": n_ar, "step_ms": m["step_ms"], "per_gpu_hbm_floor_ms": ideal_ms,
                      "non_hbm_us_per_allreduce_upper_bound": (m["step_ms"] - ideal_ms) * 1e3 / n_ar,
                      "note": "upper bound: all time above the per-GPU HBM floor (grid barriers, attention, exchange) divided by the allreduce count"}
    if extra_params:
        line["config"]["engine_params"] = extra_params
    from substratus_b200.engine import load_library

    line["engine"] = load_library().ssb_version().decode()  # names the SSB_LIB_VARIANT build, if one was selected
    if B == 1 and not args.no_batch32:  # the metric is quoted at batch 1 AND 32: same engine, second measurement
        try:
            m32 = measure(cx, eng, cfg["vocab_size"], 32, max(2, args.steps // 2), 2)
            line["batch32"] = {"value": m32["value"], "unit": "tokens/s", "e2e": m32["e2e"], "ttft_ms_p50": m32["ttft_ms_p50"],
                               "decode_ms_per_step": m32["step_ms"], "bytes_per_step": m32["bytes_step"],
                               "hbm_roofline_frac": m32["step_gbs"] / peak_gbs}
        except Exception as ex:  # the headline line above must still be printed; the failure is reported, not hidden
            line["batch32"] = {"error": repr(ex)}
    eng.close()

    # ---- the other BASELINE configs, as sub-objects of the default line (headline workload, batch 1 only)
    want = set(x for x in args.extras.split(",") if x)
    do = lambda name: (not args.no_extras) and args.workload == "llama2-7b" and B == 1 and (not want or name in want)

    def guarded(key, fn, collective):
        try:
            line[key] = fn()
        except Exception as ex:
            line[key] = {"error": repr(ex)}
        if collective and world > 1:
            cx.barrier()

    if world == 1:
        if do("gguf13b"):
            guarded("llama2_13b_q4_gguf_b32", lambda: gguf_bench(cx, 2, 1), False)
        if do("falcon40b"):
            guarded("falcon_40b", lambda: sub_bench(cx, "falcon-40b", 1, 2, 1, "falcon-40b bf16 decode, batch 1, 512+128, TP1 (1xB200)"), False)
        if do("llama70b"):
            guarded("llama2_70b", lambda: sub_bench(cx, "llama2-70b", 1, 2, 1, "llama2-70b bf16 decode, batch 1, 512+128, TP1 (1xB200): the anchor of the TP scaling target"), False)
    else:
        if do("tp_parity"):
            guarded("tp_parity", lambda: tp_parity(cx), True)
        if do("llama70b"):
            def l70():
                r = sub_bench(cx, "llama2-70b", 1, 2, 1, f"llama2-70b bf16 decode, batch 1, 512+128, TP{world}")
                cx.barrier()
                anchor = None
                if cx.rank == 0:  # TP1 anchor on the same box, rank 0 alone (137 GB fit one B200)
                    try:
                        anchor = sub_bench(cx, "llama2-70b", 1, 2, 1, "llama2-70b TP1 anchor (rank 0 alone)", tp_world=1, extra={"tp_mega": 0})
                    except Exception as ex:
                        anchor = {"error": repr(ex)}
                    r["tp1_anchor"] = anchor
                    if anchor and "value" in anchor:
                        r["speedup_vs_tp1"] = r["value"] / anchor["value"]
                return r
            guarded("llama2_70b", l70, True)
        if do("falcon40b") and world in (2, 4):
            guarded("falcon_40b", lambda: sub_bench(cx, "falcon-40b", 1, 2, 1, f"falcon-40b bf16 decode, batch 1, 512+128, TP{world}"), True)
    if world > 1:
        cx.dist.barrier()
        cx.dist.destroy_process_group()
    if cx.rank == 0 and world == 1 and do("opt125m"):
        guarded("opt_125m_cpu_container", opt_125m_container_line, False)
    if cx.rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            r = hf_cpu_measure(cfg, 1, 0, args.ref_prompt_len, args.ref_new_tokens, batch=1)
            line["cpu_baseline"] = {"value": r["decode_tok_s"], "unit": "tokens/s", "cores": r["threads"], "kind": "reference",
                                    "sample": r["sample"] + " (the library the reference's Basaran image wraps)",
                                    "ttft_ms": r["ttft_s"] * 1e3, "model_build_s": r["build_s"]}
        except Exception as ex:  # host RAM etc.
            line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": _host_threads(), "kind": "reference",
                                    "sample": f"failed: {type(ex).__name__}: {ex}"}
    if cx.rank == 0:
        print(json.dumps(line), flush=True)


# engine default for "tp_mega" under tensor parallelism (csrc/engine.cu): 3 = persistent kernel with the push exchange
TP_MEGA_DEFAULT = 3
# dram__bytes_read.sum + dram__bytes_write.sum of one decode_mega_kernel launch (ncu --set full, profiles/)
MEGA_TRAFFIC_BYTES = {("llama2-7b", 1, 1): 13.494e9}


if __name__ == "__main__":
    main()
