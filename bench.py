#!/usr/bin/env python
"""bench.py — Llama-3-8B int4 g128 QuantLinear stack on B200: bs=1 decode tok/s + 2048-token prefill TFLOP/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is ONE decode token through the hot path: the 224 GPTQ QuantLinear forwards of Llama-3-8B
(32 layers x q,k,v,o,gate,up,down; BASELINE.json configs[1]) on synthetic packed weights, chained
h -> q -> o -> gate -> down -> next layer (k, v, up are computed from the same inputs, their outputs unused: the
reference owns no attention / norm code, SURVEY.md §1).  3.63 GB of weights are streamed per step, far more than
the 126 MB L2, so no flush is needed between timed steps.  The prefill figure (M = 2048 through the same 224
layers) is measured in the same run and reported under "prefill".
With --gpus N > 1 the stack is tensor-parallel (column shards for q,k,v,gate,up; row shards + one NCCL
all-reduce for o and down), strong scaling.

--impl reference times the reference's own CPU path for this hot path (TorchAtenLinear's int4pack fused op,
restated in oracle/gptq_oracle.py::CpuFusedLinear) on the host cores; each step is a bounded sample
(1 of the 32 decoder layers).

--dump-outputs DIR writes, after the timed steps, the last hidden state of the last decode step (decode.npy) and of the
last prefill pass (prefill.npy) as float32.  Weights and inputs are seeded, so runs with the same arguments compute the
same thing and two builds can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "W4A16 g128 QuantLinear: decode tok/s + prefill TFLOPS vs HBM/TC roofline"
CFG = dict(name="Llama-3-8B", hidden=4096, inter=14336, kv=1024, layers=32, bits=4, group_size=128)
LINEARS = [  # name, K, N, parallel style
    ("q_proj", "hidden", "hidden", "col"), ("k_proj", "hidden", "kv", "col"), ("v_proj", "hidden", "kv", "col"),
    ("o_proj", "hidden", "hidden", "row"), ("gate_proj", "hidden", "inter", "col"),
    ("up_proj", "hidden", "inter", "col"), ("down_proj", "inter", "hidden", "row"),
]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops_burst=d["bf16_tflops"],
                    tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback")


def load_traffic():
    """DRAM bytes measured by ncu (--set full) for one decode launch, as a ratio of its algorithmic bytes."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(p):
        return json.load(open(p))
    return None


def algorithmic_bytes(K, N, gs, bits, M):
    G = K // gs
    return K * N * bits // 8 + G * N * 2 + G * (N * bits // 32) * 4 + M * K * 2 + M * N * 2


def make_input(M, hidden, seed, device):
    """Activations of one pass [M, hidden] fp16, seeded like the weights (synth_layer): the same in every run.
    Drawn on the device in fp32 and then cast, like the unseeded inputs before: a decode input copied in from the host
    instead measured 0.4% slower decode (B200, 1000 W power limit)."""
    gen = torch.Generator(device=device).manual_seed(seed)
    return (torch.randn(M, hidden, device=device, generator=gen) * 0.5).to(torch.float16)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each [rows, cols] host array as <out_dir>/<name>.npy in float32.  When they would exceed DUMP_BYTES in all,
    every array keeps every k-th row only, with the smallest k that fits: k follows from the shapes alone, so the sample
    is the same in every run."""
    def nbytes(k):
        return sum(4 * -(-a.shape[0] // k) * a.shape[1] for a in arrays.values())

    k = 1
    while nbytes(k) > DUMP_BYTES:
        k += 1
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a[::k].float().numpy())


# ----------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.02)

    def result(self):
        s = sorted(self.samples)
        return dict(sm_mhz=(s[len(s) // 2] if s else None), sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons),
                    samples=len(s))


# ----------------------------------------------------------------------------------------------------
def synth_layer(K, N, seed, device, bits=4, gs=128, perm=None, asym=False):
    """Random int4 codes + scales sized so activations stay O(1) through the 224-layer chain (sym, zero=8).
    perm: act-order (config 3): g_idx = (arange // gs)[perm].  asym (config 5): zero-points alternate 7 / 9 per column (a
    real qzeros tensor the kernels must decode; the weights stay zero-mean so the chained activations stay finite)."""
    gen = torch.Generator(device=device).manual_seed(seed)
    # codes uniform in 1..15: zero-mean around the symmetric zero-point 8 (a non-zero weight mean would be amplified
    # ~sqrt(K) per layer and overflow fp16 after a few of the 224 chained layers)
    qw = torch.zeros((K * bits // 32, N), dtype=torch.int32, device=device)
    for j in range(8):
        qw |= torch.randint(1, 16, (K // 8, N), dtype=torch.int32, device=device, generator=gen) << (4 * j)
    G = K // gs
    zword = (0x97979797 - (1 << 32)) if asym else (0x88888888 - (1 << 32))
    qz = torch.full((G, N * bits // 32), zword, dtype=torch.int32, device=device)
    base = 1.0 / (18.67 * K) ** 0.5  # var(q-8) = 18.67 for codes uniform in 1..15
    sc = ((0.8 + 0.4 * torch.rand(G, N, device=device, generator=gen)) * base).to(torch.float16)
    gi = torch.arange(K, dtype=torch.int32, device=device) // gs
    if perm is not None:
        gi = gi[perm.to(device).long()].contiguous()
    return dict(qweight=qw, qzeros=qz, scales=sc, g_idx=gi, bias=None, bits=bits, group_size=gs)


def build_stack(device, rank, world, layers, fuse=True, cfg=None, desc_act=False, shard=None):
    """cfg: model dims (default Llama-3-8B).  desc_act: act-order g_idx, one permutation per (layer, input) — q/k/v and
    gate/up of a GPTQ checkpoint share theirs (same input Hessian).  shard=(r, w): build rank r's TP-w shards without a
    process group (per-GPU work of a larger TP job, no collective)."""
    from gptqmodel_b200 import B200QuantLinear, fuse_siblings, tp

    cfg = cfg or CFG
    sr, sw = shard if shard is not None else (rank, world)
    stack = []
    for li in range(layers):
        mods = {}
        perms = {}
        for j, (name, kk, nn_, style) in enumerate(LINEARS):
            K, N = cfg[kk], cfg[nn_]
            perm = None
            if desc_act:
                pk = {"q_proj": "h", "k_proj": "h", "v_proj": "h", "gate_proj": "h2", "up_proj": "h2"}.get(name, name)
                if pk not in perms:
                    perms[pk] = torch.randperm(K, generator=torch.Generator().manual_seed(li * 8 + len(perms)))
                perm = perms[pk]
            L = synth_layer(K, N, seed=li * 16 + j, device=device, gs=cfg["group_size"], perm=perm)
            if sw > 1:
                if style == "col" or desc_act:   # act-order row layers are served column-parallel (tp.GatheredColumnParallelLinear)
                    L = tp.shard_columns(L, sr, sw)
                else:
                    L = tp.shard_rows(L, sr, sw)
            m = B200QuantLinear.from_checkpoint_tensors(L["qweight"], L["qzeros"], L["scales"], L["g_idx"], cfg["bits"],
                                                        cfg["group_size"], desc_act=desc_act, device=device)
            mods[name] = m
            del L
        if fuse:
            # q/k/v and gate/up consume the same activations: one decode launch each (b2q_decode_multi)
            fuse_siblings([mods["q_proj"], mods["k_proj"], mods["v_proj"]])
            fuse_siblings([mods["gate_proj"], mods["up_proj"]])
        stack.append(mods)
    torch.cuda.empty_cache()
    return stack


P2P_AR = None  # optional gptqmodel_b200.tp.P2PAllReduce (--p2p-allreduce): our one-shot kernel over NVLink peer memory


FUSED_AR = None  # optional gptqmodel_b200.tp.FusedDecodeAllReduce (--fused-allreduce, experimental): matmul + all-reduce in one launch


_RP_CACHE = {}


def _row_parallel(mod, x, world):
    """o_proj / down_proj: the library's row-parallel wrapper (gptqmodel_b200.tp.RowParallelLinear): shard matmul + ONE
    all-reduce — the fused launch / our peer-memory kernel for decode-sized outputs, NCCL overlapped with the next token
    block's GEMM for prefill-sized ones."""
    if world == 1:
        return mod(x)
    rp = _RP_CACHE.get(id(mod))
    if rp is None:
        from gptqmodel_b200 import tp as _tp
        rp = _tp.RowParallelLinear(mod, reduce=FUSED_AR if FUSED_AR is not None else P2P_AR,
                                   overlap_chunks=OVERLAP_CHUNKS)
        _RP_CACHE[id(mod)] = rp
    return rp(x)


OVERLAP_CHUNKS = 1


def _all_reduce(t):
    import torch.distributed as dist

    if P2P_AR is not None and t.numel() <= P2P_AR.max_elems:
        P2P_AR(t)
    else:
        dist.all_reduce(t)


def run_stack(stack, h, world):
    """One pass of the hot path over a batch h [M, hidden]; returns the last hidden state."""
    for mods in stack:
        a = mods["q_proj"](h)
        mods["k_proj"](h)
        mods["v_proj"](h)
        h2 = _row_parallel(mods["o_proj"], a, world)
        g = mods["gate_proj"](h2)
        mods["up_proj"](h2)
        h = _row_parallel(mods["down_proj"], g, world)
    return h


def capture(stack, x_static, world):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            run_stack(stack, x_static, world)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = run_stack(stack, x_static, world)
    return g, out


def timed_replays(g, n, world, device):
    import torch.distributed as dist

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms = float(t.item())
    return ms


# ----------------------------------------------------------------------------------------------------
def cpu_layer(seed=0):
    """One decoder layer (7 QuantLinears) on the reference's CPU fused path."""
    import oracle

    mods = []
    for j, (name, kk, nn_, _style) in enumerate(LINEARS):
        K, N = CFG[kk], CFG[nn_]
        L = synth_layer(K, N, seed=seed * 16 + j, device="cpu")
        mods.append((name, oracle.CpuFusedLinear(L["qweight"], L["qzeros"], L["scales"], L["g_idx"], 4, 128)))
    return dict(mods)


def cpu_layer_step(mods, h):
    a = mods["q_proj"].forward(h)
    mods["k_proj"].forward(h)
    mods["v_proj"].forward(h)
    h2 = mods["o_proj"].forward(a)
    g = mods["gate_proj"].forward(h2)
    mods["up_proj"].forward(h2)
    return mods["down_proj"].forward(g)


CPU_DISTINCT_LAYERS = 4  # 4 x 109 MB of int4pack weights: the rotation exceeds any host LLC, like a real token's 3.6 GB stream


class CpuArm:
    """The reference's CPU path for this hot path (TorchAtenLinear int4pack op, restated in oracle/), timed so that the
    number is reproducible (VERDICT r01 weak #8): CPU_DISTINCT_LAYERS distinct decoder layers are rotated so every step
    streams its weights from DRAM, the thread count is chosen by the MEDIAN of >= 10 steps per candidate, and the result
    is the median step with its p10-p90 spread."""

    def __init__(self):
        self.layers = [cpu_layer(seed=s) for s in range(CPU_DISTINCT_LAYERS)]
        self.h = (torch.randn(1, CFG["hidden"]) * 0.5).to(torch.float16)
        self.i = 0
        self.thread_table = {}

    def step(self):
        t0 = time.perf_counter()
        cpu_layer_step(self.layers[self.i % len(self.layers)], self.h)
        self.i += 1
        return time.perf_counter() - t0

    def pick_threads(self, iters=10):
        ncpu = os.cpu_count() or 1
        cands = sorted({c for c in (4, 8, 16, 32, 64, 128, ncpu // 2, ncpu) if 1 <= c <= ncpu})
        best = (None, 1e30)
        for c in cands:
            torch.set_num_threads(c)
            first = self.step()
            if first > 20 * best[1]:  # oversubscribed (measured: 0.8 ms per layer at 64 threads, 480 ms at 128): stop here
                self.thread_table[c] = round(first * 1e3, 3)
                break
            ts = sorted(self.step() for _ in range(iters))
            med = ts[len(ts) // 2]
            self.thread_table[c] = round(med * 1e3, 3)
            if med < best[1]:
                best = (c, med)
        torch.set_num_threads(best[0])
        return best[0]

    def measure(self, steps, warmup):
        for _ in range(max(warmup, 1)):
            self.step()
        ts = sorted(self.step() for _ in range(steps))
        n = len(ts)
        med = ts[n // 2]
        return dict(median=med, p10=ts[max(0, int(0.1 * n))], p90=ts[min(n - 1, int(0.9 * n))], steps=n)

    def describe(self, r):
        return (f"each step = 1 decoder layer (7 QuantLinears, M=1) of {CPU_DISTINCT_LAYERS} distinct layers in rotation "
                f"(weights from DRAM, not LLC) through the restated TorchAtenLinear path "
                f"(aten::_weight_int4pack_mm_for_cpu); {r['steps']} timed steps, median {r['median'] * 1e3:.2f} ms/layer "
                f"(p10 {r['p10'] * 1e3:.2f}, p90 {r['p90'] * 1e3:.2f}); tok/s = 1/(32 * median); threads chosen by the "
                f"median of 10 steps per candidate: {self.thread_table} ms/layer")


def workload_name(n_lin, Mp):
    # ONE string for both arms (the driver compares config.workload of the b200 and the reference arm)
    return (f"{CFG['name']} int4 g128 sym QuantLinear stack ({n_lin} linears): bs=1 decode step "
            f"(value) + {Mp}-token prefill pass (prefill.*)")


def time_cpu_baseline(budget_s=15.0):
    arm = CpuArm()
    arm.pick_threads()
    probe = arm.measure(5, 1)
    steps = int(max(10, min(400, budget_s / max(probe["median"], 1e-4))))
    r = arm.measure(steps, 1)
    return 1.0 / (r["median"] * CFG["layers"]), arm, r


def reference_arm(args, rank):
    if rank != 0:
        return
    arm = CpuArm()
    arm.pick_threads()
    r = arm.measure(args.steps, args.warmup)  # exactly K timed steps; the value is their median
    per_layer = r["median"]
    toks = 1.0 / (per_layer * CFG["layers"])
    n_lin = len(LINEARS) * CFG["layers"]
    line = {
        "impl": "reference", "metric": METRIC, "value": toks, "unit": "tok/s", "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": args.warmup, "ms_per_step": per_layer * CFG["layers"] * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16 (aten int4pack CPU kernel)",
        "data": "synthetic",
        "config": {"workload": workload_name(n_lin, args.prefill_tokens), "parallelism": "cpu",
                   "note": "reference arm: the decode step only, on the host cores"},
        "cpu_baseline": {"value": toks, "unit": "tok/s", "cores": torch.get_num_threads(), "kind": "port",
                         "spread_tok_s": [1.0 / (r["p90"] * CFG["layers"]), 1.0 / (r["p10"] * CFG["layers"])],
                         "sample": arm.describe(r)},
        "e2e": {"value": toks, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


CFG70 = dict(name="Llama-3-70B", hidden=8192, inter=28672, kv=1024, layers=80, bits=4, group_size=128)
MIXTRAL = dict(name="Mixtral-8x7B", hidden=4096, inter=14336, kv=1024, layers=32, experts=8, top_k=2, bits=4, group_size=64)


def time_stack(stack, M, world, device, iters, hidden, runner=None):
    """ms per pass of `stack` over M tokens (whole pass in one CUDA graph, CUDA events, max over ranks)."""
    x = (torch.randn(M, hidden, device=device) * 0.5).to(torch.float16)
    run = runner or run_stack
    s_ = torch.cuda.Stream()
    s_.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s_):
        for _ in range(2):
            run(stack, x, world)
    torch.cuda.current_stream().wait_stream(s_)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = run(stack, x, world)
    for _ in range(3):
        g.replay()
    ms = timed_replays(g, iters, world, device) / iters
    fin = bool(torch.isfinite(out).all())
    del g
    return ms, fin


def stack_bytes_and_weights(cfg, layers, shard_world=1, M=1):
    sizes = [(cfg[kk] // (shard_world if st == "row" else 1), cfg[nn_] // (shard_world if st == "col" else 1))
             for _, kk, nn_, st in LINEARS]
    alg = sum(algorithmic_bytes(K, N, cfg["group_size"], 4, M) for K, N in sizes) * layers
    weights = sum(K * N for K, N in sizes) * layers
    return alg, weights


def build_mixtral(device, rank, world, layers, shard=None):
    """Mixtral-8x7B int4 g64 ASYMMETRIC (BASELINE configs[4]): per layer q|k|v, o and the 8-expert MoE block (w1 / w3 column-,
    w2 row-sharded, every rank holds a slice of every expert), experts through the GROUPED kernels (no host sync)."""
    from gptqmodel_b200 import B200QuantLinear, fuse_siblings, moe, tp

    c = MIXTRAL
    sr, sw = shard if shard is not None else (rank, world)
    mk = lambda L: B200QuantLinear.from_checkpoint_tensors(L["qweight"], L["qzeros"], L["scales"], L["g_idx"], 4,  # noqa: E731
                                                           c["group_size"], sym=False, device=device)
    col = (lambda L: tp.shard_columns(L, sr, sw)) if sw > 1 else (lambda L: L)
    row = (lambda L: tp.shard_rows(L, sr, sw)) if sw > 1 else (lambda L: L)
    gen = torch.Generator().manual_seed(0)
    stack = []
    for li in range(layers):
        sl = lambda K, N, j: synth_layer(K, N, seed=li * 64 + j, device=device, gs=c["group_size"], asym=True)  # noqa: E731
        q, k, v = (mk(col(sl(c["hidden"], n, j))) for j, n in enumerate((c["hidden"], c["kv"], c["kv"])))
        o = mk(row(sl(c["hidden"], c["hidden"], 3)))
        fuse_siblings([q, k, v])
        w1 = [mk(col(sl(c["hidden"], c["inter"], 4 + 3 * e))) for e in range(c["experts"])]
        w3 = [mk(col(sl(c["hidden"], c["inter"], 5 + 3 * e))) for e in range(c["experts"])]
        w2 = [mk(row(sl(c["inter"], c["hidden"], 6 + 3 * e))) for e in range(c["experts"])]
        blk = moe.MoEExperts(w1, w3, w2, grouped=True)
        logits = torch.randn(2048, c["experts"], generator=gen)
        ids, w = moe.route_topk(logits, c["top_k"])
        stack.append(dict(q=q, k=k, v=v, o=o, moe=blk, ids=ids.to(device), w=w.to(device)))
    torch.cuda.empty_cache()
    return stack


def run_mixtral(stack, h, world):
    M = h.shape[0]
    for L in stack:
        a = L["q"](h)
        L["k"](h)
        L["v"](h)
        h2 = _row_parallel(L["o"], a, world)
        h = L["moe"](h2, L["ids"][:M], L["w"][:M])   # ends in the block's single all-reduce when world > 1
    return h


def extra_workloads(args, device, rank, world, peaks):
    """BASELINE configs 3-5 and the batched-decode regime, measured in the same run (VERDICT r01 missing #6)."""
    extra = {}
    hbm = peaks["hbm_gbs"]

    def entry(name, fn):
        t0 = time.perf_counter()
        try:
            extra[name] = fn()
        except Exception as e:  # noqa: BLE001
            extra[name] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
        torch.cuda.empty_cache()
        if rank == 0:
            print(f"[bench] extra.{name}: {time.perf_counter() - t0:.1f} s", file=sys.stderr, flush=True)

    if world == 1:
        def act_order():
            st = build_stack(device, 0, 1, CFG["layers"], fuse=True, desc_act=True)
            alg, weights = stack_bytes_and_weights(CFG, CFG["layers"])
            alg += 4 * sum(CFG[kk] for _, kk, _, _ in LINEARS) * CFG["layers"]   # + g_idx / perm reads
            ms, fin = time_stack(st, 1, 1, device, 20, CFG["hidden"])
            msp, _ = time_stack(st, args.prefill_tokens, 1, device, 3, CFG["hidden"])
            return {"workload": "Llama-3-8B int4 g128 act-order (desc_act=True; q|k|v and gate|up share their g_idx), "
                                "1xB200 (BASELINE configs[2])", "decode_tok_s": 1e3 / ms,
                    "decode_frac_hbm": alg / (ms * 1e-3) / 1e9 / hbm,
                    "prefill_tflops": 2.0 * args.prefill_tokens * weights / (msp * 1e-3) / 1e12, "finite": fin}
        entry("act_order_8b", act_order)

    def small_batch(stack):
        out = {}
        for M in (16, 64):
            alg, _ = stack_bytes_and_weights(CFG, args.layers, world, M)
            ms, fin = time_stack(stack, M, world, device, 10, CFG["hidden"])
            out[f"M{M}"] = {"ms_per_step": ms, "tokens_per_s": M * 1e3 / ms, "frac_hbm": alg / (ms * 1e-3) / 1e9 / hbm,
                            "finite": fin}
        out["workload"] = "the same Llama-3-8B stack at 16 / 64 tokens per step (batched / speculative decode: small-batch tier)"
        return out
    extra["_small_batch_fn"] = small_batch

    if world in (1, 8):
        def l70():
            shard = None if world == 8 else (0, 8)
            st = build_stack(device, rank, world, CFG70["layers"], fuse=True, cfg=CFG70, shard=shard)
            alg, weights = stack_bytes_and_weights(CFG70, CFG70["layers"], 8)
            ms, fin = time_stack(st, 1, world, device, 10, CFG70["hidden"])
            msp, _ = time_stack(st, args.prefill_tokens, world, device, 2, CFG70["hidden"])
            return {"workload": "Llama-3-70B int4 g128, TP-8 (BASELINE configs[3])" + (
                        "" if world == 8 else ": ONE rank's shard stack on one GPU, no all-reduce (per-GPU work only)"),
                    "decode_tok_s": 1e3 / ms, "decode_frac_hbm_per_gpu": alg / (ms * 1e-3) / 1e9 / hbm,
                    "prefill_tflops_per_gpu": 2.0 * args.prefill_tokens * weights / (msp * 1e-3) / 1e12,
                    "prefill_ms": msp, "finite": fin}
        entry("llama3_70b_tp8", l70)

    if world in (1, 4):
        def mixtral():
            c = MIXTRAL
            shard = None if world == 4 else (0, 4)
            st = build_mixtral(device, rank, world, c["layers"], shard=shard)
            # bytes per token per GPU: attention linears + the top-2 active experts (SURVEY 8d: 6.80 GB per token / 4)
            att = sum(algorithmic_bytes(K, N, 64, 4, 1) for K, N in (
                (c["hidden"], c["hidden"] // 4), (c["hidden"], c["kv"] // 4), (c["hidden"], c["kv"] // 4),
                (c["hidden"] // 4, c["hidden"])))
            exp = c["top_k"] * (2 * algorithmic_bytes(c["hidden"], c["inter"] // 4, 64, 4, 1) +
                                algorithmic_bytes(c["inter"] // 4, c["hidden"], 64, 4, 1))
            alg = (att + exp) * c["layers"]
            ms, fin = time_stack(st, 1, world, device, 10, c["hidden"], runner=run_mixtral)
            ms8, _ = time_stack(st, 8, world, device, 5, c["hidden"], runner=run_mixtral)
            return {"workload": "Mixtral-8x7B int4 g64 asym, TP-4, experts through gptqmodel_b200.moe.MoEExperts (one token: "
                                "decode-tier MoE launches, 8 tokens: grouped small-batch kernels) "
                                "(BASELINE configs[4])" + ("" if world == 4 else
                                                           ": ONE rank's shard stack on one GPU, no all-reduce"),
                    "decode_tok_s": 1e3 / ms, "decode_frac_hbm_per_gpu": alg / (ms * 1e-3) / 1e9 / hbm,
                    "decode_bytes_per_token_per_gpu": alg, "batch8_tokens_per_s": 8e3 / ms8, "finite": fin}
        entry("mixtral_8x7b_tp4", mixtral)
    return extra


# ----------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--prefill-tokens", type=int, default=2048)
    ap.add_argument("--prefill-iters", type=int, default=0, help="0 = auto")
    ap.add_argument("--layers", type=int, default=CFG["layers"], help="debug: fewer layers (result marked invalid)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra workloads (BASELINE configs 3-5, batched decode)")
    ap.add_argument("--no-competitors", action="store_true", help="skip the same-box Marlin comparison")
    ap.add_argument("--with-vllm", action="store_true", help="competitors: also vLLM's Marlin build (import takes ~70 s)")
    ap.add_argument("--nccl-allreduce", action="store_true",
                    help="keep NCCL for the small decode all-reduces (default: b2q_allreduce, our one-shot kernel over "
                         "NVLink peer memory; measured 715 vs 605 tok/s at TP-4)")
    ap.add_argument("--overlap-chunks", type=int, default=1,
                    help="N > 1 prefill: token blocks whose all-reduce overlaps the next block's GEMM (default 1 = off: "
                         "measured SLOWER at TP-4, 17.5 vs 12.3 ms per pass, profiles/r02_tp_notes.md)")
    ap.add_argument("--no-fuse", action="store_true", help="one launch per QuantLinear (224/step) instead of fusing q/k/v and gate/up")
    ap.add_argument("--decode-v2", action="store_true",
                    help="EXPERIMENTAL: decode tier v2 (b2q_decode2.cu; sets B2Q_DECODE_V2=1), result marked experimental")
    ap.add_argument("--fused-allreduce", action="store_true",
                    help="EXPERIMENTAL (N > 1): row-parallel matmul + all-reduce in one launch (b2q_decode_allreduce)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last decode step's and prefill pass's outputs to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    global OVERLAP_CHUNKS
    OVERLAP_CHUNKS = args.overlap_chunks
    if args.decode_v2:
        os.environ["B2Q_DECODE_V2"] = "1"

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank)
        return
    if world != args.gpus:
        if args.gpus == 1 and world == 1:
            pass
        else:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    peaks = load_peaks()
    if world > 1 and not args.nccl_allreduce:
        from gptqmodel_b200 import tp as _tp

        global P2P_AR
        try:
            P2P_AR = _tp.P2PAllReduce(device, max_elems=8 * CFG["hidden"])
        except Exception as e:  # noqa: BLE001  (symmetric memory unavailable: NCCL carries the all-reduce)
            if rank == 0:
                print(f"[bench] P2PAllReduce unavailable ({type(e).__name__}: {e}); using NCCL", file=sys.stderr)
            P2P_AR = None

    if world > 1 and args.fused_allreduce:
        from gptqmodel_b200 import tp as _tp

        global FUSED_AR
        FUSED_AR = _tp.FusedDecodeAllReduce(device, max_elems=8 * CFG["hidden"])

    _t0 = time.perf_counter()

    def phase(msg):
        if rank == 0:
            print(f"[bench +{time.perf_counter() - _t0:6.1f}s] {msg}", file=sys.stderr, flush=True)

    stack = build_stack(device, rank, world, args.layers, fuse=not args.no_fuse)
    phase("stack built")
    hidden = CFG["hidden"]
    sizes = [(CFG[kk] // (world if st == "row" else 1), CFG[nn_] // (world if st == "col" else 1))
             for _, kk, nn_, st in LINEARS]
    n_lin = len(LINEARS) * args.layers
    alg_bytes_step = sum(algorithmic_bytes(K, N, 128, 4, 1) for K, N in sizes) * args.layers  # per GPU
    weights_total = sum(CFG[kk] * CFG[nn_] for _, kk, nn_, _ in LINEARS) * args.layers

    # ---------------- decode: kernel-resident timing (inputs already in HBM) ----------------
    x_static = make_input(1, hidden, seed=1, device=device)
    g_dec, out_dec = capture(stack, x_static, world)
    for _ in range(args.warmup):
        g_dec.replay()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms = timed_replays(g_dec, args.steps, world, device)
    clocks_dec = None
    ms_per_step = ms / args.steps
    toks = 1e3 / ms_per_step
    finite = bool(torch.isfinite(out_dec).all())

    # ---------------- decode e2e: host buffers, H2D + graph + D2H every step ----------------
    x_host = x_static.cpu().pin_memory()
    y_host = torch.empty(1, hidden, dtype=torch.float16).pin_memory()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        x_static.copy_(x_host, non_blocking=True)
        g_dec.replay()
        y_host.copy_(out_dec, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_toks = args.steps / e2e_s

    phase("decode timed")
    # ---------------- prefill: M tokens through the same 224 layers ----------------
    Mp = args.prefill_tokens
    xp = make_input(Mp, hidden, seed=2, device=device)
    g_pre, out_pre = capture(stack, xp, world)
    it_pre = args.prefill_iters or max(3, min(args.steps, 10))
    for _ in range(3):
        g_pre.replay()
    ms_pre = timed_replays(g_pre, it_pre, world, device) / it_pre
    sampler.stop_flag = True
    sampler.join(timeout=2)
    clocks = sampler.result()
    flops = 2.0 * Mp * weights_total
    tflops = flops / (ms_pre * 1e-3) / 1e12
    # e2e prefill: tokens' activations from pinned host memory + result back
    xp_host = xp.cpu().pin_memory()
    yp_host = torch.empty(Mp, hidden, dtype=torch.float16).pin_memory()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(it_pre):
        xp.copy_(xp_host, non_blocking=True)
        g_pre.replay()
        yp_host.copy_(out_pre, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    pre_e2e_ms = (time.perf_counter() - t0) / it_pre * 1e3

    phase("prefill timed")
    if args.dump_outputs and rank == 0:
        # the host copies of the last decode step and prefill pass: what a caller of the timed path receives
        dump_outputs(args.dump_outputs, {"decode": y_host, "prefill": yp_host})
        phase(f"outputs written to {args.dump_outputs}")
    # ---------------- the other BASELINE configs + batched decode + competitor kernels ----------------
    extra, competitors = {}, None
    if not args.no_extra and args.layers == CFG["layers"]:
        extra = extra_workloads(args, device, rank, world, peaks)
        sb = extra.pop("_small_batch_fn")
        try:
            extra["small_batch"] = sb(stack)
        except Exception as e:  # noqa: BLE001
            extra["small_batch"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    phase("extra workloads done")
    if rank == 0 and world == 1 and not args.no_competitors and args.layers == CFG["layers"]:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import competitors as _comp

            arms = ("b2q", "marlin_ref", "marlin_vllm") if args.with_vllm else ("b2q", "marlin_ref")
            competitors = _comp.run(arms, Ms=(1, 16, 64, 2048), nlayers=CFG["layers"], stack=True, verbose=False)
            competitors["note"] = ("same box, same packed checkpoint tensors; marlin_ref = the reference's own "
                                   "gptqmodel_ext/marlin compiled for sm_100a by baseline/build_marlin.py; per-shape us = "
                                   "mean over a CUDA graph walking >= 600 MB of distinct layers; stack = 224 separate "
                                   "launches per step for every arm (this repo's headline additionally fuses q|k|v and gate|up)")
        except Exception as e:  # noqa: BLE001
            competitors = {"error": f"{type(e).__name__}: {str(e)[:300]}"}

    phase("competitors done")
    # ---------------- CPU baseline (rank 0, N=1 only) ----------------
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, arm, r = time_cpu_baseline()
        cpu_base = {"value": v, "unit": "tok/s", "cores": torch.get_num_threads(), "kind": "port",
                    "spread_tok_s": [1.0 / (r["p90"] * CFG["layers"]), 1.0 / (r["p10"] * CFG["layers"])],
                    "sample": arm.describe(r)}
        del arm

    phase("cpu baseline done")
    if rank == 0:
        achieved = alg_bytes_step / (ms_per_step * 1e-3) / 1e9  # GB/s per GPU
        tr = load_traffic()
        n_launch = n_lin if args.no_fuse else 4 * args.layers
        traffic = (tr["decode_kernel"]["ratio"] * alg_bytes_step / n_launch) if tr else None
        line = {
            "metric": METRIC, "value": toks, "unit": "tok/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {
                "workload": workload_name(n_lin, Mp),
                "parallelism": f"tp{world}" + ("" if world == 1 else
                                               (", decode all-reduce: b2q_allreduce (P2P one-shot kernel), "
                                                "prefill all-reduce: NCCL" if P2P_AR is not None
                                                else ", all-reduce: NCCL")),
                "l2": "3.63 GB of distinct weights per step >> 126 MB L2: no flush needed between timed steps",
                "timing": "CUDA graph of the whole step, CUDA events around K replays, max over ranks",
                **({"experimental": [f for f, on in (("decode-v2", args.decode_v2),
                                                     ("fused-allreduce", FUSED_AR is not None)) if on]}
                   if (args.decode_v2 or FUSED_AR is not None) else {}),
            },
            "roofline": {
                "kernel": ("decode2_kernel (EXPERIMENTAL b2q_decode2.cu: deferred tile epilogue, warp groups); "
                           if args.decode_v2 else
                           "decode tier (fragment-major int4 -> mma.sync, per-warp bulk-copy rings, PDL): decode2_kernel for "
                           "the multi-tile q|k|v and gate|up launches, decode_kernel for o_proj / down_proj; ")
                          + ("one launch per QuantLinear" if args.no_fuse else
                             "q/k/v and gate/up siblings share a launch: 4 launches per decoder layer"),
                "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "peak_source": peaks["source"],
                "algorithmic_bytes_per_launch": alg_bytes_step / n_launch,
                "traffic": None if args.decode_v2 else traffic,  # the ncu capture is of the default kernel
                "traffic_note": "average per launch = measured DRAM/algorithmic ratio of the ncu --set full capture "
                                "(profiles/r02_decode_ncu.txt: 30,317,568 B DRAM vs 30,539,776 B algorithmic for the "
                                "4096x14336 launch) x algorithmic bytes per launch",
            },
            "prefill": {
                "tokens": Mp, "ms_per_pass": ms_pre, "tflops": tflops, "iters": it_pre,
                "tokens_per_s": Mp / (ms_pre * 1e-3),
                "roofline": {"kernel": "gemm2p_kernel (persistent CTA pairs, tcgen05.mma.cta_group::2 + TMA, TMEM accumulators)", "bound": "tensor",
                             "achieved": tflops / world, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                             "frac": tflops / world / peaks["tflops_sustained"],
                             "peak_note": "sustained cuBLAS bf16 (kernel timed inside a long step); burst peak "
                                          f"{peaks['tflops_burst']}",
                             "traffic": (tr or {}).get("gemm2p_kernel", {}).get("dram_bytes"),
                             "traffic_note": "DRAM bytes of ONE 4096x4096 M=2048 launch (ncu --set full, "
                                             "profiles/r02_gemm2p_ncu.txt); tensor-bound kernel"},
                "e2e_ms_per_pass": pre_e2e_ms,
                "e2e_tokens_per_s": Mp / (pre_e2e_ms * 1e-3),
            },
            "e2e": {"value": e2e_toks, "unit": "tok/s", "h2d_bytes_per_step": hidden * 2,
                    "d2h_bytes_per_step": hidden * 2,
                    "how": "pinned host x -> H2D -> graph replay of the 224 forward() calls -> D2H -> stream sync"},
            "gpu_launches": n_lin if args.no_fuse else 4 * args.layers,
            "clocks": clocks,
            "finite_outputs": finite,
        }
        if extra:
            line["extra"] = extra
        if competitors is not None:
            line["competitors"] = competitors
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        if args.layers != CFG["layers"]:
            line["invalid"] = f"debug run with {args.layers} layers"
        print(json.dumps(line))
    if world > 1:
        # Tearing an NCCL process group down while captured CUDA graphs still hold its kernels hangs in
        # destroy_process_group (seen on the 2-GPU box): drop the graphs, sync, and leave without the destroy.
        del g_dec, g_pre
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
