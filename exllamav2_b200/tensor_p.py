"""Tensor parallelism over the column shard -- the multi-GPU row of SURVEY.md 8(e).

Mirror of exllamav2/tensor_p.py (TPContext, :102-181 split tables) + the TP forward loops of ext_qattn.cpp:261-732 /
ext_qmlp.cpp:326-473, re-designed for one process per GPU:

  * every linear is split on OUTPUT columns exactly as ExLlamaV2Linear.tp_split does (linear.py:567-587; see
    linear.tp_column_slice) -- q/k/v by head, gate/up by intermediate column, o_proj / down_proj by hidden column,
    lm_head by vocab column.  A shard is cut from the checkpoint tensors BEFORE make_q_matrix, so a rank only ever holds
    (and re-packs) its own columns.  GPTQ shards the same way (the reference rejects it, ext_qmatrix.cpp:130-135).
  * the K/V cache is sharded by kv-head (cache.py:659-692): attention is rank-local.
  * a sharded activation is re-replicated with ONE all-gather (torch.distributed, NCCL over NVLink) where the reference
    stages through pinned host memory (ext_tp.cpp:129-293): after attention (rows x H*hd), after O-proj into the residual
    stream, after act*mul (rows x intermediate), after down-proj -- 4 per layer + 1 for the logits.  No all-reduce: the
    summation order of every output element is the single-GPU order, results are bit-identical to the unsharded run.
  * the whole sharded decode step, collectives included, is captured in one CUDA graph per rank.

At batch 1 these collectives are latency-bound (8-22 KB each); DESIGN.md discusses the peer-store epilogue that replaces
them next.  Host-side logic (split tables, slicing, gather layout) runs on CPU tensors over gloo in tests/test_tp_gloo.py.
"""
from __future__ import annotations

import json
import math
import os
import time

import torch
import torch.distributed as dist


def split_even(n: int, world: int, multiple: int) -> list[tuple[int, int]]:
    """[a, b) column range per rank: equal shares, each a multiple of `multiple` (tensor_p.py:120-158 uses head_dim for
    attention, 128 for the MLP intermediate, 32 for hidden / vocab; scale nibbles force a multiple of 8)."""
    if n % (world * multiple):
        raise ValueError(f"cannot split {n} columns over {world} ranks in multiples of {multiple}")
    step = n // world
    return [(r * step, (r + 1) * step) for r in range(world)]


class TPContext:
    """Split tables of one model for `world` ranks (tensor_p.py:14-18: KV heads, Q heads, ID intermediate, RS hidden, VC vocab)."""

    def __init__(self, cfg, rank: int, world: int):
        self.rank, self.world = rank, world
        hd = cfg.head_dim
        if cfg.num_kv_heads % world or cfg.num_heads % world:
            raise ValueError(f"{cfg.num_kv_heads} kv heads / {cfg.num_heads} heads do not split over {world} ranks")
        self.kv = split_even(cfg.num_kv_heads * hd, world, hd)
        self.q = split_even(cfg.num_heads * hd, world, hd)
        self.id = split_even(cfg.intermediate_size, world, 8)
        self.rs = split_even(cfg.hidden_size, world, 32)
        self.vc = split_even(cfg.vocab_size, world, 32)

    def mine(self, table):
        return table[self.rank]

    # -- collectives ------------------------------------------------------------------------------------------------
    def all_gather_cols(self, full: torch.Tensor, local: torch.Tensor, scratch: torch.Tensor | None = None):
        """full[rows, N] <- concat over ranks of local[rows, N / world] along columns.  `local` may be the rank's own
        column slice of `full` (in place).  rows == 1: a column concat IS a contiguous concat (one all-gather straight
        into `full`); rows > 1: gather into [world, rows, N/world] scratch and de-block."""
        rows, n = full.shape
        nl = n // self.world
        if self.world == 1:
            if local.data_ptr() != full.data_ptr():
                full.copy_(local)
            return
        if rows == 1:
            flat = full.view(-1)
            src = flat[self.rank * nl:(self.rank + 1) * nl]
            if local.data_ptr() != src.data_ptr():
                src.copy_(local.view(-1))
            _all_gather_flat(flat, src)
            return
        if scratch is None:
            scratch = torch.empty((self.world, rows, nl), dtype=full.dtype, device=full.device)
        mine = scratch[self.rank]
        mine.copy_(local)
        _all_gather_flat(scratch.view(-1), mine.view(-1))
        full.view(rows, self.world, nl).copy_(scratch.transpose(0, 1))


def _all_gather_flat(out_flat: torch.Tensor, in_flat: torch.Tensor):
    if dist.get_backend() == "nccl":
        dist.all_gather_into_tensor(out_flat, in_flat)
    else:                                   # gloo (CPU tests): list form
        n = in_flat.numel()
        parts = [torch.empty_like(in_flat) for _ in range(dist.get_world_size())]
        dist.all_gather(parts, in_flat.clone())
        for r, p in enumerate(parts):
            out_flat[r * n:(r + 1) * n].copy_(p)


def tp_column_slice_t(w: dict, a: int, b: int) -> dict:
    """torch version of linear.tp_column_slice: columns [a, b) of an EXL2 / GPTQ tensor dict (linear.py:567-587)."""
    assert a % 8 == 0 and b % 8 == 0
    out = dict(w)
    if "q_weight" in w:
        out["q_weight"] = w["q_weight"][:, a:b].contiguous()
        out["q_scale"] = w["q_scale"][:, a // 8:b // 8].contiguous()
    else:
        out["qweight"] = w["qweight"][:, a:b].contiguous()
        out["qzeros"] = w["qzeros"][:, a // 8:b // 8].contiguous()
        out["scales"] = w["scales"][:, a:b].contiguous()
    if "bias" in w:
        out["bias"] = w["bias"][a:b].contiguous()
    return out


class ExLlamaV2DecoderTP:
    """Column-sharded twin of model.ExLlamaV2Decoder: same synthetic weights (same seeds, generated in full and cut), one
    rank's shard of every linear and of the Q4 cache."""

    def __init__(self, cfg, rank: int, world: int, device, seed: int = 0, batch_size: int = 1, cache_len: int | None = None):
        from . import ext as ext_c
        from . import synthetic
        from .ext import none_tensor
        from .linear import ExLlamaV2Linear
        from .model import ExLlamaV2Cache_Q4, LlamaConfig, rope_tables
        self.ext = ext_c
        self.cfg, self.device = cfg, torch.device(device)
        self.tp = tp = TPContext(cfg, rank, world)
        dev = self.device
        H, KVH, hd, hid, inter = cfg.num_heads, cfg.num_kv_heads, cfg.head_dim, cfg.hidden_size, cfg.intermediate_size
        self.Hl, self.KVHl = H // world, KVH // world
        self.inter_l = inter // world
        gen = torch.Generator(device=dev)
        gen.manual_seed(seed)
        self.weight_bytes = 0
        self.layers, self.linears = [], []

        def lin(K, N, plan, s, cols, perm_seed=None):
            w = synthetic.random_linear(K, N, plan, device=dev, seed=s, weight_std=1.0 / math.sqrt(K), perm_seed=perm_seed)
            a, b = cols
            ws = tp_column_slice_t(w, a, b)
            del w
            self.weight_bytes += synthetic.algorithmic_bytes(ws, 1)
            l = ExLlamaV2Linear(K, b - a, device=dev)
            l.load(ws)
            self.linears.append(l)
            return l

        class _L:
            pass

        s = seed * 100003
        for li in range(cfg.num_layers):
            L = _L()
            mp = cfg.plan.mlp[li % len(cfg.plan.mlp)]
            # same tensors as model.ExLlamaV2Decoder (k / v share q's permutation, up shares gate's)
            L.q_proj = lin(hid, H * hd, cfg.plan.attn, s + 1, tp.mine(tp.q), s + 1)
            L.k_proj = lin(hid, KVH * hd, cfg.plan.attn, s + 2, tp.mine(tp.kv), s + 1)
            L.v_proj = lin(hid, KVH * hd, cfg.plan.attn, s + 3, tp.mine(tp.kv), s + 1)
            L.o_proj = lin(H * hd, hid, cfg.plan.attn, s + 4, tp.mine(tp.rs))
            L.gate = lin(hid, inter, mp, s + 5, tp.mine(tp.id), s + 5)
            L.up = lin(hid, inter, mp, s + 6, tp.mine(tp.id), s + 5)
            L.down = lin(inter, hid, mp, s + 7, tp.mine(tp.rs))
            s += 16
            L.input_norm = (1 + 0.1 * torch.randn((hid,), device=dev, generator=gen)).half()
            L.post_norm = (1 + 0.1 * torch.randn((hid,), device=dev, generator=gen)).half()
            L.temp_a = torch.empty((64, self.inter_l), dtype=torch.half, device=dev)
            L.temp_b = torch.empty((64, self.inter_l), dtype=torch.half, device=dev)
            # rank-local blocks: this rank's heads / intermediate columns; o_proj and down are applied as column shards below
            L.attn = ext_c.make_q_attn(L.input_norm, none_tensor, True, False, cfg.norm_eps, L.q_proj.q_handle, L.k_proj.q_handle,
                                       L.v_proj.q_handle, 0, none_tensor, none_tensor, 64, hid, self.Hl, self.KVHl, hd,
                                       cfg.max_seq_len, True, 2, hd, none_tensor, none_tensor, none_tensor, none_tensor, False, True)
            L.mlp = ext_c.make_q_mlp(L.post_norm, none_tensor, True, cfg.norm_eps, L.gate.q_handle, L.up.q_handle, 0,
                                     none_tensor, L.temp_a, none_tensor, none_tensor, 64, False, True, none_tensor, none_tensor,
                                     False, True)
            self.layers.append(L)
        self.final_norm = (1 + 0.1 * torch.randn((hid,), device=dev, generator=gen)).half()
        self.lm_head = lin(hid, cfg.vocab_size, cfg.plan.head, s + 9, tp.mine(tp.vc))
        self.embed = (0.02 * torch.randn((cfg.vocab_size, hid), device=dev, generator=gen)).half()
        cache_len = cache_len or min(cfg.max_seq_len, 1024)
        self.sin, self.cos = rope_tables(hd, max(cfg.max_seq_len, (cache_len + 255) // 256 * 256), cfg.rope_theta, dev)
        local_cfg = LlamaConfig(cfg.name, hid, inter, self.Hl, self.KVHl, hd, cfg.num_layers, cfg.vocab_size, cfg.max_seq_len)
        self.cache = ExLlamaV2Cache_Q4(local_cfg, batch_size, cache_len, dev)        # this rank's kv heads
        self.batch_size = B = batch_size
        self.ids = torch.zeros((B, 1), dtype=torch.long, device=dev)
        self.x = torch.empty((B, hid), dtype=torch.half, device=dev)
        self.q = torch.empty((B, 1, self.Hl * hd), dtype=torch.half, device=dev)
        self.k = torch.empty((B, 1, self.KVHl * hd), dtype=torch.half, device=dev)
        self.v = torch.empty_like(self.k)
        self.attn_full = torch.empty((B, H * hd), dtype=torch.half, device=dev)
        self.act_full = torch.empty((B, inter), dtype=torch.half, device=dev)
        self.xn = torch.empty((B, hid), dtype=torch.half, device=dev)
        self.logits = torch.empty((B, cfg.vocab_size), dtype=torch.half, device=dev)
        self.graph = None
        self.pos = 0

    def _forward_rows(self, x, q, k, v, q_len: int):
        """x [rows, hidden] replicated on every rank; rows = B * q_len."""
        e, cfg, tp, cache = self.ext, self.cfg, self.tp, self.cache
        B, hd = self.batch_size, cfg.head_dim
        rows = x.shape[0]
        a0, a1 = tp.mine(tp.q)
        r0, r1 = tp.mine(tp.rs)
        i0, i1 = tp.mine(tp.id)
        attn_full = self.attn_full if rows == self.attn_full.shape[0] else torch.empty((rows, cfg.num_heads * hd), dtype=torch.half, device=x.device)
        act_full = self.act_full if rows == self.act_full.shape[0] else torch.empty((rows, cfg.intermediate_size), dtype=torch.half, device=x.device)
        for li, L in enumerate(self.layers):
            e.q_attn_forward_1(L.attn, x, B, q_len, -1, cache.cache_seqlens, q, k, v, self.sin, self.cos)
            attn_l = attn_full[:, a0:a1] if rows == 1 else torch.empty((rows, a1 - a0), dtype=torch.half, device=x.device)
            e.paged_attn_decode_q4(q.view(B, q_len, self.Hl, hd), k.view(B, q_len, self.KVHl, hd), v.view(B, q_len, self.KVHl, hd),
                                   cache.key_states[li], cache.key_scales[li], cache.value_states[li], cache.value_scales[li],
                                   cache.cache_seqlens, cache.block_table, attn_l.view(B, q_len, self.Hl, hd), 1.0 / math.sqrt(hd))
            tp.all_gather_cols(attn_full, attn_l)
            e.gemm_half_q_half_accum(attn_full, L.o_proj.q_handle, x[:, r0:r1])       # my hidden columns: x += attn @ Wo[:, cols]
            tp.all_gather_cols(x, x[:, r0:r1])
            act_l = act_full[:, i0:i1] if rows == 1 else L.temp_a[:rows]
            e.q_mlp_forward_gateup(L.mlp, x, act_l)
            tp.all_gather_cols(act_full, act_l)
            e.gemm_half_q_half_accum(act_full, L.down.q_handle, x[:, r0:r1])
            tp.all_gather_cols(x, x[:, r0:r1])
        cache.cache_seqlens.add_(q_len)

    def _decode_step(self):
        torch.index_select(self.embed, 0, self.ids.view(-1), out=self.x)
        self._forward_rows(self.x, self.q, self.k, self.v, 1)
        self.ext.rms_norm(self.x, self.final_norm, self.xn, self.cfg.norm_eps)
        v0, v1 = self.tp.mine(self.tp.vc)
        if self.batch_size == 1:
            self.ext.gemm_half_q_half(self.xn, self.lm_head.q_handle, self.logits[:, v0:v1], False)
            self.tp.all_gather_cols(self.logits, self.logits[:, v0:v1])
        else:
            loc = torch.empty((self.batch_size, v1 - v0), dtype=torch.half, device=self.x.device)
            self.ext.gemm_half_q_half(self.xn, self.lm_head.q_handle, loc, False)
            self.tp.all_gather_cols(self.logits, loc)

    def prefill(self, ids: torch.Tensor, chunk: int = 8):
        B, T = ids.shape
        hd = self.cfg.head_dim
        if self.pos + T > self.cache.max_seq_len:
            raise RuntimeError(f"prompt of {T} tokens does not fit the K/V cache")
        self.pos += T
        for t0 in range(0, T, chunk):
            n = min(chunk, T - t0)
            x = self.embed[ids[:, t0:t0 + n]].reshape(B * n, -1).contiguous()
            q = torch.empty((B, n, self.Hl * hd), dtype=torch.half, device=self.device)
            k = torch.empty((B, n, self.KVHl * hd), dtype=torch.half, device=self.device)
            self._forward_rows(x, q, k, torch.empty_like(k), n)

    def capture(self, body=None):
        body = body or self._decode_step
        # the warm-up step and the capture run on a side stream over the decoder's static buffers: everything already queued on the
        # caller's stream (earlier decode steps whose results the caller may not have read yet) has to be finished first
        torch.cuda.synchronize()
        s = torch.cuda.Stream(self.device)
        saved = self.cache.cache_seqlens.clone()
        with torch.cuda.stream(s):
            body()
            torch.cuda.synchronize()
            self.cache.cache_seqlens.copy_(saved)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                body()
        torch.cuda.synchronize()
        self.cache.cache_seqlens.copy_(saved)
        self.graph = g
        return g

    def decode(self, ids: torch.Tensor) -> torch.Tensor:
        if self.pos + 1 > self.cache.max_seq_len:
            raise RuntimeError(f"K/V cache is full ({self.pos} of {self.cache.max_seq_len} positions)")
        self.pos += 1
        self.ids.copy_(ids)
        if self.graph is not None:
            self.graph.replay()
        else:
            self._decode_step()
        return self.logits


# ---- bench.py --gpus N > 1 ------------------------------------------------------------------------------------------

def run_bench(args, rank: int, world: int, metric: str, unit: str):
    """One process per GPU (torchrun): sharded decode, CUDA-event timing, max over ranks, rank 0 prints the JSON line."""
    from . import ext as ext_c
    from .model import PRESETS
    import bench as bench_mod                     # ClockSampler / measured_peaks live in bench.py
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    cfg = PRESETS[args.model]()
    t_build = time.time()
    dec = ExLlamaV2DecoderTP(cfg, rank, world, dev, seed=0, batch_size=1, cache_len=1024)
    torch.cuda.synchronize()
    t_build = time.time() - t_build
    g = torch.Generator(device="cpu").manual_seed(0)
    prompt = torch.randint(0, cfg.vocab_size, (1, args.prompt_len), generator=g).to(dev)
    dec.prefill(prompt)
    dec.ids.copy_(prompt[:, -1:])
    torch.cuda.synchronize()
    dist.barrier()

    def step_with_argmax():
        dec._decode_step()
        torch.argmax(dec.logits, dim=-1, keepdim=True, out=dec.ids)

    l0 = ext_c.launch_count()
    captured = True
    try:
        graph = dec.capture(step_with_argmax)
        launches_per_step = (ext_c.launch_count() - l0) // 2
        run = graph.replay
    except Exception as ex:                     # NCCL refused capture: run the same step eagerly
        captured = False
        torch.cuda.synchronize()
        l0 = ext_c.launch_count()
        step_with_argmax()
        launches_per_step = ext_c.launch_count() - l0
        run = step_with_argmax
        if rank == 0:
            print(f"# graph capture of the sharded step failed ({type(ex).__name__}: {ex}); running eagerly", flush=True)
    W, K = max(3, args.warmup), args.steps
    for _ in range(W):
        run()
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with bench_mod.ClockSampler(local) as clk:
        torch.cuda.synchronize()
        e0.record()
        for _ in range(K):
            run()
        e1.record()
        torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(ms.item()) / K
    finite = bool(torch.isfinite(dec.logits).all())
    if rank == 0 and args.dump_outputs:
        bench_mod.dump_outputs(args.dump_outputs, {"logits": dec.logits, "next_token": dec.ids})

    # e2e: host token in, host logits out, every step (rank 0's host feeds all ranks through a broadcast of the id)
    ids_host = torch.zeros((1, 1), dtype=torch.long).pin_memory()
    logits_host = torch.empty((1, cfg.vocab_size), dtype=torch.half).pin_memory()
    plain = dec.capture() if captured else None
    def e2e_step():
        dec.ids.copy_(ids_host, non_blocking=True)
        dist.broadcast(dec.ids, src=0)
        if plain is not None:
            plain.replay()
        else:
            dec._decode_step()
        logits_host.copy_(dec.logits, non_blocking=True)
        torch.cuda.synchronize()
        ids_host[0, 0] = int(torch.argmax(logits_host.float(), dim=-1)[0])
    for _ in range(3):
        e2e_step()
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        e2e_step()
    t_e2e = torch.tensor([(time.perf_counter() - t0) / K], device=dev)
    dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    t_e2e = float(t_e2e.item())

    wb = torch.tensor([float(dec.weight_bytes)], device=dev)
    dist.all_reduce(wb)
    if rank == 0:
        peak, peak_src = bench_mod.measured_peaks()
        achieved = float(wb.item()) / world / (ms_per_step * 1e-3) / 1e9
        line = {
            "metric": metric, "value": 1000.0 / ms_per_step, "unit": unit, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "fp16 (int2-8 weights, fp32 accumulate)", "data": "synthetic",
            "config": {"workload": f"{cfg.name} single-stream decode, {args.prompt_len}-token prompt, Q4 KV cache, bs=1, tensor-parallel column shard over {world} GPUs",
                       "l2": "inputs_exceed_l2 (weights streamed once per step)", "parallelism": f"tp{world}",
                       "collectives_per_step": 4 * cfg.num_layers + 1, "graph": captured, "build_s": round(t_build, 1), "finite": finite},
            "clocks": clk.summary(),
            "e2e": {"value": 1.0 / t_e2e, "unit": unit, "h2d_bytes_per_step": 8, "d2h_bytes_per_step": cfg.vocab_size * 2, "ms_per_step": t_e2e * 1e3},
            "gpu_launches": int(launches_per_step * K * world), "launches_per_step": int(launches_per_step),
            "roofline": {"bound": "hbm", "kernel": "gemv_i8_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "peak_source": peak_src,
                         "note": "per-GPU algorithmic weight bytes / whole step time (collectives and attention included): a lower bound on the kernel's own rate"},
            "cpu_baseline": None,
        }
        print(json.dumps(line), flush=True)
    # Leave without tearing NCCL down: destroying a communicator that live CUDA graphs still reference blocks forever
    # (seen on 2 x B200, torch 2.11 / NCCL 2.28); the process is at its end anyway.
    torch.cuda.synchronize()
    dist.barrier()
    import sys
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)
