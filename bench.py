#!/usr/bin/env python
"""
bench.py — headline benchmark of the DeTikZify hot path on B200 (contract in the task brief, tier ④).

Workload (BASELINE.json configs[1], named in ``config.workload``): detikzify-ds-1.3b shape, random-init
bf16 weights, ONE synthetic 384x384 figure per GPU, batch-1 greedy generation: ViT encode + concat-3
projector + 243-token image-prefix prefill, then KV-cached single-token decode with the fused sampler
up to a total length of 2048 (1805 new tokens). One "step" = one such figure.

  value  = decoded tokens/s, whole job (sum over GPUs), pixels already resident in HBM, the decode loop
           enqueued as one CUDA-graph launch per token with NO per-token host synchronisation.
  e2e    = the same metric through the public API ``model.generate()``: pixel_values start in pinned
           host memory (H2D inside the timed region) and every generated token is read back by the host
           (the streamer/stopping-criteria contract of the reference) before the next one is consumed.
  roofline = algorithmic HBM bytes of the decode steps (weights once per token + KV read at the running
           context; dtk_decode_bytes) / CUDA-event time of the decode region, vs MEASURED_PEAKS.json.
  cpu_baseline = the oracle (HF Llama+SigLIP wired like the reference; oracle/hf_oracle.py) on the host cores,
           bounded sample, through stock HF ``generate`` (BASELINE.md section 2 protocol).
  ds7b     = BASELINE.json configs[3]/[4] shape as extra keys (detikzify-ds-7b random-init): batch-1 decode roofline, and
           figure-sharded rollouts (8 figures per rank, 32 nucleus-sampled rollouts per figure forked off one prefilled
           prompt, results gathered once) — tokens/s over all ranks, max-over-ranks device time.

``--impl reference`` times that CPU path alone (the reference package itself is pure Python glue over
HF modules and does not import offline; see DESIGN.md): HF ``generate(do_sample=False, max_new_tokens=n)`` incl. ViT
and the 243-token prefill, fp32 and bf16 probed in the warm-up, thread count = scheduler affinity capped by the cgroup
quota.
Multi-GPU: figures are independent -> one engine per rank, ONE NCCL broadcast of the weight arena at
load, no per-step collective; scaling is weak (one figure per GPU per step); every rank is pinned to the NUMA node of
its GPU.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="nllg/detikzify-ds-1.3b")
    ap.add_argument("--total-len", type=int, default=2048)
    ap.add_argument("--cpu-tokens", type=int, default=64, help="new tokens of the bounded CPU sample inside our arm")
    ap.add_argument("--ref-tokens", type=int, default=256, help="new tokens per step of --impl reference (BASELINE.md: 256)")
    ap.add_argument("--no-7b", action="store_true", help="skip the ds-7b (configs[3]/[4]) block")
    ap.add_argument("--figures-per-rank", type=int, default=8)
    ap.add_argument("--rollouts", type=int, default=32)
    ap.add_argument("--rollout-tokens", type=int, default=128)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-vit-sweep", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed paths computed in their last step to DIR/<name>.npy (float32 / float64)")
    return ap.parse_args()


def dump_outputs(out_dir: str, arrays: dict):
    """Last-step outputs of the timed paths as DIR/<name>.npy: floats as float32, token ids as float64 (exact). Same
    arguments -> same seeded inputs, so two builds can be compared output for output. Whole-array unless noted; a
    larger output is a fixed, seeded sample (<= 64 MB in all)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        if torch.is_tensor(t):
            t = t.detach()
            a = (t.float() if t.is_floating_point() else t).cpu().numpy()
        else:
            a = np.asarray(t)
        a = a.astype(np.float32 if a.dtype.kind == "f" else np.float64)
        total += a.nbytes
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    assert total <= 64 << 20, total


def seeded_sample(t: torch.Tensor, n: int, seed: int = 0) -> torch.Tensor:
    """A fixed, seeded sample of n elements of t (all of t when it is not larger)."""
    flat = t.reshape(-1)
    if flat.numel() <= n:
        return flat
    idx = torch.randint(flat.numel(), (n,), generator=torch.Generator().manual_seed(seed)).sort().values
    return flat[idx.to(flat.device)]


# ---------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of ``kernel`` from the committed `ncu --set full` capture
    (profiles/r*_ncu_full_<kernel>.json, written by tools/ncu_summary.py); None when no capture is committed."""
    best = None
    for f in sorted((ROOT / "profiles").glob(f"r*_ncu_full_{kernel}.json")):
        try:
            d = json.loads(f.read_text())
            best = {"bytes_per_launch": d["dram_bytes_read"] + d["dram_bytes_write"], "ctx": d.get("ctx"), "source": f"profiles/{f.name}"}
        except (OSError, ValueError, KeyError):
            continue
    return best


# ---------------------------------------------------------------------------------- CPU reference arm
def synthetic_pixels(batch: int, image_size: int, seed: int = 1000) -> torch.Tensor:
    """pixel_values = 2*U[0,1)-1 (range of the (x-0.5)/0.5 normalisation), SURVEY.md section 8d."""
    out = []
    for i in range(batch):
        g = torch.Generator().manual_seed(seed + i)
        out.append(2 * torch.rand(3, image_size, image_size, generator=g) - 1)
    return torch.stack(out)


class _Stamps:
    """HF streamer protocol: records when the prompt and every new token reach the host."""

    def __init__(self):
        self.t = []

    def put(self, value):
        self.t.append(time.perf_counter())

    def end(self):
        pass


class CpuArm:
    """The reference's HF CPU path as closely as this container allows (oracle/hf_oracle.py: stock HF Llama + SigLIP wired
    like detikzify/model/v1/modeling_detikzify.py). One step = one figure through stock ``GenerationMixin.generate``
    (greedy, n new tokens) incl. ViT + projector + 243-token prefill; decode tokens/s is taken between the first and the
    last new token as seen by a streamer (prefill excluded, as on the GPU arm's ``value``)."""

    def __init__(self, model_name: str):
        from detikzify_b200.model.configuration import preset
        from detikzify_b200.model.weights import random_init
        from detikzify_b200.parallel import host_threads
        self.threads = host_threads()
        # all usable host threads, also under torchrun (which exports OMP_NUM_THREADS=1 to its workers)
        torch.set_num_threads(int(os.environ.get("DTK_CPU_THREADS", self.threads["use"])))
        self.cores = torch.get_num_threads()
        self.cfg = preset(model_name)
        self.sd = random_init(self.cfg, seed=0)
        self.oracles = {}
        self.pix = synthetic_pixels(1, self.cfg.vision_config.image_size)
        self.ids = torch.full((1, self.cfg.num_patches), self.cfg.patch_token_id, dtype=torch.long)

    def oracle(self, dtype):
        from oracle.hf_oracle import Oracle
        if dtype not in self.oracles:
            self.oracles[dtype] = Oracle(self.cfg.to_dict(), self.sd, dtype=dtype)
        return self.oracles[dtype]

    def figure(self, dtype, n_new: int):
        """-> dict(total_s, vit_s, prefill_s, decode_tok_s)"""
        o = self.oracle(dtype)
        P = self.cfg.num_patches
        st = _Stamps()
        t0 = time.perf_counter()
        img = o.image_embeds(self.pix)
        t1 = time.perf_counter()
        embeds = o.spliced_embeds(self.ids, img)
        with torch.no_grad():
            out = o.llm.generate(input_ids=self.ids, inputs_embeds=embeds, bad_words_ids=[[o.image_token_id]],
                                 max_length=P + n_new, min_length=P + n_new, do_sample=False, streamer=st,
                                 pad_token_id=self.cfg.pad_token_id)
        t2 = time.perf_counter()
        new = [t for t in st.t if t > t1]
        # st.t[0] is the prompt (or absent with inputs_embeds); new tokens follow
        first, last = new[-n_new], new[-1]
        assert out.shape[1] >= n_new
        return {"total_s": t2 - t0, "vit_s": t1 - t0, "prefill_s": first - t1, "decode_tok_s": (n_new - 1) / max(last - first, 1e-9)}


def cpu_reference(model_name: str, n_new: int, steps: int, warmup: int, probe_tokens: int = 12):
    """Bounded CPU sample. The warm-up probes fp32 and bf16 (reference scripts load bf16; fp32 is often faster on CPU) and
    the faster dtype runs the timed steps. Returns (summary dict for the JSON line, CpuArm)."""
    arm = CpuArm(model_name)
    probe = {}
    for dt in (torch.float32, torch.bfloat16):
        try:
            probe[str(dt).split(".")[-1]] = arm.figure(dt, probe_tokens)
        except Exception as e:  # a dtype the CPU kernels do not support
            probe[str(dt).split(".")[-1]] = {"error": repr(e)[:120]}
    ok = {k: v for k, v in probe.items() if "decode_tok_s" in v}
    best = max(ok, key=lambda k: ok[k]["decode_tok_s"])
    dtype = getattr(torch, best)
    # keep one step near 40 s at most
    n = max(16, min(n_new, int(40.0 * ok[best]["decode_tok_s"])))
    for _ in range(max(0, warmup - 1)):
        arm.figure(dtype, n)
    runs = [arm.figure(dtype, n) for _ in range(steps)]
    tps = [r["decode_tok_s"] for r in runs]
    mean = sum(tps) / len(tps)
    sd = (sum((x - mean) ** 2 for x in tps) / len(tps)) ** 0.5
    return {
        "value": mean, "stdev": sd, "dtype": best, "new_tokens": n, "runs": runs, "probe": probe,
        "cores": arm.cores, "threads": arm.threads,
        "sec_per_step": sum(r["total_s"] for r in runs) / len(runs),
    }, arm


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r, arm = cpu_reference(args.model, args.ref_tokens, steps=args.steps, warmup=max(1, args.warmup))
    P = arm.cfg.num_patches
    sample = (f"per step: 1 figure through stock HF generate(do_sample=False): ViT ({r['runs'][0]['vit_s']:.2f}s) + {P}-token prefill "
              f"({r['runs'][0]['prefill_s']:.2f}s) + {r['new_tokens']} greedy tokens at ctx {P}..{P + r['new_tokens']}, {r['dtype']} weights, "
              f"{r['cores']} threads (affinity {r['threads']['affinity']}, cgroup quota {r['threads']['cgroup_quota']}, host {r['threads']['host_logical']}); "
              f"value = decode tokens/s between first and last new token, mean of {args.steps} steps (stdev {r['stdev']:.2f}); "
              f"probe fp32 {r['probe'].get('float32', {}).get('decode_tok_s', 'n/a')} / bf16 {r['probe'].get('bfloat16', {}).get('decode_tok_s', 'n/a')} tok/s")
    line = {
        "impl": "reference", "metric": "TikZ tokens/sec/GPU (decode, 384px cond, 2k ctx)", "value": r["value"], "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["sec_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32" if r["dtype"] == "float32" else "bf16", "data": "synthetic",
        "config": {"workload": f"{args.model} random-init, 1x384px synthetic figure, batch-1 greedy generate (bounded CPU sample)"},
        "cpu_baseline": {"value": r["value"], "unit": "tokens/s", "cores": r["cores"], "kind": "port", "sample": sample,
                         "stdev": r["stdev"], "vit_s": r["runs"][0]["vit_s"], "prefill_s": r["runs"][0]["prefill_s"]},
        "e2e": {"value": r["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))

    from detikzify_b200.model import load
    from detikzify_b200.parallel import gather_results, pin_to_gpu_numa, shard
    numa = pin_to_gpu_numa(local)

    model, processor = load(args.model, device_map=local, torch_dtype=torch.bfloat16, broadcast=world > 1, seed=0)
    cfg, eng = model.config, model.engine
    dev = model.device
    P, total = cfg.num_patches, min(args.total_len, eng.max_len)
    n_new = total - P
    ids = torch.full((P,), cfg.patch_token_id, dtype=torch.int64, device=dev)
    pix_host = synthetic_pixels(1, cfg.vision_config.image_size, seed=1000 + rank).pin_memory()
    pix_dev = pix_host.to(dev)
    # greedy, EOS suppressed for the throughput run so every figure decodes the full 1805 tokens (SURVEY §8d)
    params = eng.sampling(do_sample=False, bad_token=cfg.image_token_id, begin_suppress_token=-1)
    stream = torch.cuda.Stream(device=dev)
    slot = eng.seq_alloc()

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def figure(timed: bool):
        """ViT -> projector -> prefill -> first token -> (n_new - 1) graph-launched decode+sample steps."""
        if timed:
            ev[0].record(stream)
        img = eng.image_embeds(pix_dev)[0]
        last, _ = eng.prefill(slot, ids, 0, img, 0)
        first, _ = eng.sample(last, params, suppress=[0])
        tok0 = int(first.item())
        eng.gen_begin([slot], [P], [tok0], params)
        if timed:
            ev[1].record(stream)
        for _ in range(n_new - 1):
            eng.gen_step()
        if timed:
            ev[2].record(stream)
        out = eng.gen_wait(n_new - 2)  # last token has landed on the host
        eng.gen_end()
        return {"image_embeds": img, "prefill_logits": last, "tokens": [tok0, *out]}

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            figure(False)
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        launches0 = eng.launch_count
        t_all = t_dec = 0.0
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(stream)
        dec_ms = []
        dump = {}
        for _ in range(args.steps):
            dump = figure(True)
            stream.synchronize()
            dec_ms.append(ev[1].elapsed_time(ev[2]))
        stop.record(stream)
        barrier()
        t_all = start.elapsed_time(stop) / 1e3
        t_dec = sum(dec_ms) / 1e3
        launches = eng.launch_count - launches0
        clocks = sampler.stop() if rank == 0 else None

        # ---- e2e through the public API (host buffers, per-token host visibility)
        e2e_t = None
        if not args.no_e2e:
            from detikzify_b200.util.generation import TokenStreamer
            ids_host = ids.cpu()[None]

            def api_figure():
                st = TokenStreamer()
                out = model.generate(input_ids=ids_host, pixel_values=pix_host, bad_words_ids=[[cfg.image_token_id]],
                                     begin_suppress_tokens=[cfg.eos_token_id], streamer=st, do_sample=False,
                                     max_length=total, eos_token_id=-1)
                assert out.shape[1] == total, out.shape
                return out
            model._img_cache = None
            api_figure()  # warm-up (graph capture for this sampling config)
            barrier()
            s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                model._img_cache = None      # a new figure every step: ViT + full prefill inside the timed region
                model._slot_tokens = []
                dump["e2e_sequences"] = api_figure()
            torch.cuda.synchronize()
            e2e_t = time.perf_counter() - t0
            barrier()

        # ---- secondary metric of BASELINE.json ("ViT encode ms/img", configs[2]: batch sweep @384px), rank 0 only
        vit = None
        if rank == 0 and not args.no_vit_sweep:
            vit = {}
            v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for B in (1, 8, 64):
                pix_b = synthetic_pixels(B, cfg.vision_config.image_size, seed=7).to(dev)
                for _ in range(2):
                    eng.vit_encode(pix_b)
                reps = 5 if B < 64 else 3
                v0.record(stream)
                for _ in range(reps):
                    tokens, pooled = eng.vit_encode(pix_b)
                v1.record(stream)
                stream.synchronize()
                vit[str(B)] = v0.elapsed_time(v1) / reps / B
                dump[f"vit_b{B}_pooled"], dump[f"vit_b{B}_tokens_sample"] = pooled, seeded_sample(tokens, 1 << 16)
                del pix_b
        barrier()

    # ---- BASELINE.json configs[3] / configs[4] shape: detikzify-ds-7b, figures striped over the ranks, 32 nucleus-sampled
    # rollouts per figure forked off one prefilled 243-token image prompt. Extra keys; the headline stays configs[1].
    ds7b = None
    t7 = torch.zeros(3, dtype=torch.float64)
    bytes_dec = sum(eng.decode_bytes(P + 1 + i) for i in range(n_new - 1))   # (taken before the engine may be released)
    persistent = eng.get_option("decode_persistent") == 1
    eng.seq_free(slot)
    if not args.no_7b:
        del model, eng
        torch.cuda.empty_cache()
        R, F, NT7 = args.rollouts, args.figures_per_rank, args.rollout_tokens
        name7 = "nllg/detikzify-ds-7b"
        model7, _ = load(name7, device_map=local, torch_dtype=torch.bfloat16, broadcast=world > 1, seed=0, device_init=True,
                         max_seqs=R + 1, max_batch=R)
        e7, c7 = model7.engine, model7.config
        P7 = c7.num_patches
        figures = shard(list(range(F * world)), rank, world)           # global figure indices of this rank (striped)
        pix7 = torch.cat([synthetic_pixels(1, c7.vision_config.image_size, seed=5000 + g) for g in figures]).to(dev)
        ids7 = torch.full((P7,), c7.patch_token_id, dtype=torch.int64, device=dev)
        slots7 = [e7.seq_alloc() for _ in range(R)]
        nuc = e7.sampling(temperature=0.8, top_p=0.95, do_sample=True, bad_token=c7.image_token_id, begin_suppress_token=-1, seed=3)
        grd = e7.sampling(do_sample=False, bad_token=c7.image_token_id, begin_suppress_token=-1)
        with torch.cuda.stream(stream):
            # (a) batch-1 decode at ctx 512 on the persistent kernel
            ctx7 = 512
            warm_ids = torch.randint(0, 30000, (ctx7,), generator=torch.Generator().manual_seed(1)).to(dev)
            e7.prefill(slots7[0], warm_ids, 0, None, 0)
            tok1 = torch.tensor([5], device=dev)
            for _ in range(3):
                e7.decode([slots7[0]], [ctx7], tok1)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            for _ in range(10):
                logits7 = e7.decode([slots7[0]], [ctx7], tok1)
            a1.record(stream)
            stream.synchronize()
            b1_ms = a0.elapsed_time(a1) / 10

            def figure7(fi: int):
                """ViT + projector + prefill of figure fi, fork to R rollouts, NT7 sampled tokens each -> [R] last tokens"""
                img = e7.image_embeds(pix7[fi:fi + 1])[0]
                for sl in slots7[1:]:
                    e7.seq_share(slots7[0], sl, 0)            # release the previous figure's prefix
                last, _ = e7.prefill(slots7[0], ids7, 0, img, 0)
                for sl in slots7[1:]:
                    e7.seq_share(slots7[0], sl, P7)           # rollouts READ the image prefix from slot 0 (no copy)
                first, _ = e7.sample(last[None].expand(R, -1).contiguous(), nuc, suppress=[0] * R, steps=[0] * R, seq_ids=list(range(R)))
                e7.gen_begin(slots7, [P7] * R, [int(t) for t in first.tolist()], nuc, list(range(R)))
                for _ in range(NT7 - 1):
                    e7.gen_step()
                out = e7.gen_wait(NT7 - 2)
                e7.gen_end()
                return out

            figure7(0)                                                    # warm-up (graph capture)
            barrier()
            l0 = e7.launch_count
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record(stream)
            local_out = [figure7(fi) for fi in range(len(figures))]
            g1.record(stream)
            barrier()
            roll_s = g0.elapsed_time(g1) / 1e3
            dump["ds7b_b1_decode_logits"] = logits7
            dump["ds7b_rollout_last_tokens"] = local_out
            launches7 = e7.launch_count - l0
        gathered = gather_results([(g, o[:4]) for g, o in zip(figures, local_out)])   # one gather at the end (examples/eval.py:132)
        t7 = torch.tensor([b1_ms, roll_s, float(len(gathered))], dtype=torch.float64)
        kvb = e7.decode_bytes(1) - e7.decode_bytes(0)
        ds7b_local = {"decode_bytes_ctx512": e7.decode_bytes(ctx7), "weights_bytes": e7.decode_bytes(0), "kv_bytes_per_pos": kvb,
                      "launches": int(launches7), "persistent": e7.get_option("decode_persistent") == 1}
        for sl in reversed(slots7):      # borrowers before the slot that lends them the image prefix
            e7.seq_free(sl)
    barrier()

    # max over ranks
    vals = torch.tensor([t_all, t_dec, e2e_t or 0.0, float(t7[0]), float(t7[1])], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    t_all, t_dec, e2e_t, b1_ms7, roll_s7 = vals.tolist()
    if rank == 0 and not args.no_7b:
        R, F, NT7 = args.rollouts, args.figures_per_rank, args.rollout_tokens
        peak7, _src = peaks()
        d = ds7b_local
        # rollouts: bytes per decode step = weights once + the KV every rollout reads (private copies today) and the
        # UNIQUE KV bytes (shared 243-token prefix counted once) that an ideal prefix-sharing cache would read
        steps7 = NT7 - 1
        kv_priv = sum(R * (243 + 1 + i) * d["kv_bytes_per_pos"] for i in range(steps7))
        kv_uniq = sum((243 + R * (1 + i)) * d["kv_bytes_per_pos"] for i in range(steps7))
        ds7b = {
            "model": "nllg/detikzify-ds-7b random-init bf16 (device-side init)",
            "b1_decode": {"ctx": 512, "ms_per_token": b1_ms7, "achieved_gbs": d["decode_bytes_ctx512"] / (b1_ms7 * 1e-3) / 1e9,
                          "frac_of_hbm_peak": d["decode_bytes_ctx512"] / (b1_ms7 * 1e-3) / 1e9 / peak7, "persistent_kernel": d["persistent"],
                          "note": "max over ranks, CUDA events, 10 tokens after 3 warm-up"},
            "rollouts": {"figures_per_rank": F, "figures_total": int(t7[2]) if world == 1 else F * world, "rollouts_per_figure": R, "new_tokens": NT7,
                         "sampling": "temperature 0.8, top-p 0.95", "seconds": roll_s7,
                         "tokens_per_s": world * F * R * NT7 / roll_s7, "ms_per_figure": roll_s7 / F * 1e3,
                         "includes": "ViT + projector + 243-token prefill + 31 shared-prefix borrowers (dtk_seq_share) + decode, per figure; max over ranks",
                         "roofline_unique_kv": {"bytes_per_figure": d["weights_bytes"] * steps7 + kv_uniq,
                                                "frac_of_hbm_peak": F * (d["weights_bytes"] * steps7 + kv_uniq) / roll_s7 / 1e9 / peak7},
                         "roofline_private_kv": {"bytes_per_figure": d["weights_bytes"] * steps7 + kv_priv,
                                                 "frac_of_hbm_peak": F * (d["weights_bytes"] * steps7 + kv_priv) / roll_s7 / 1e9 / peak7},
                         "gpu_launches": d["launches"]},
        }

    if rank == 0:
        new_per_step = n_new
        value = world * args.steps * new_per_step / t_all
        # roofline of the decode region (dominant: the per-token decode step = weights + KV stream)
        peak, peak_src = peaks()
        achieved = bytes_dec * args.steps / t_dec / 1e9
        kernel_name = ("decode_mega_kernel (persistent cooperative weight-streaming decode kernel, 1 launch per token) + sample_kernel"
                       if persistent else "decode step (CUDA graph: fused RMSNorm+GEMV / split-K attention / sampler kernels of one token)")
        traffic = ncu_traffic("decode_mega_kernel") if persistent else None
        line = {
            "metric": "TikZ tokens/sec/GPU (decode, 384px cond, 2k ctx)", "value": value, "unit": "tokens/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_all / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.model} random-init bf16, 1x384px synthetic figure per GPU, batch-1 greedy: ViT + projector + "
                                   f"{P}-token prefill + {n_new} decoded tokens to total length {total}",
                       "l2": "inputs larger than L2: 2.56 GB of weights streamed per token (126 MB L2)",
                       "parallelism": f"figure-sharded dp{world}, 1 NCCL weight broadcast at load, no per-step collective"},
            "roofline": {"bound": "hbm", "kernel": kernel_name,
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": peak_src, "bytes_per_token_avg": bytes_dec / (n_new - 1),
                         "decode_ms_per_token": t_dec / args.steps / (n_new - 1) * 1e3},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if vit:
            # tensor roofline of the ViT (dense contractions, SURVEY.md section 8 a2: 666 GFLOP per image at so400m/14@384)
            vc = cfg.vision_config
            n_tok = (vc.image_size // vc.patch_size) ** 2
            D, Iv, Lv = vc.hidden_size, vc.intermediate_size, vc.num_hidden_layers
            flop_img = Lv * (2 * n_tok * (4 * D * D + 2 * D * Iv) + 4 * n_tok * n_tok * D) + 2 * n_tok * D * 3 * vc.patch_size ** 2
            tpeak, tsrc = 1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s)"
            pk = ROOT / "MEASURED_PEAKS.json"
            if pk.exists() and json.loads(pk.read_text()).get("bf16_tflops_sustained"):
                tpeak, tsrc = float(json.loads(pk.read_text())["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
            best_b = min(vit, key=vit.get)
            ach = flop_img / (vit[best_b] * 1e-3) / 1e12
            line["vit_encode_ms_per_img"] = {
                "batch": vit, "note": "SigLIP-so400m/14@384 tokens + pooled output, pixels resident, CUDA events",
                "roofline": {"bound": "tensor", "gflop_per_img": flop_img / 1e9, "achieved": ach, "unit": "TFLOP/s", "at_batch": int(best_b),
                             "peak": tpeak, "frac": ach / tpeak, "peak_source": tsrc}}
        if e2e_t:
            line["e2e"] = {"value": world * args.steps * new_per_step / e2e_t, "unit": "tokens/s",
                           "h2d_bytes_per_step": int(pix_host.numel() * 4 + P * 8), "d2h_bytes_per_step": int(new_per_step * 4)}
        if ds7b:
            line["ds7b"] = ds7b
        line["host"] = {"numa": numa}
        if not args.no_cpu_baseline and world == 1:
            r, _ = cpu_reference(args.model, args.cpu_tokens, steps=1, warmup=1)
            line["cpu_baseline"] = {"value": r["value"], "unit": "tokens/s", "cores": r["cores"], "kind": "port",
                                    "sample": f"1 figure through stock HF generate: ViT ({r['runs'][0]['vit_s']:.2f}s) + {P}-token prefill ({r['runs'][0]['prefill_s']:.2f}s) + "
                                              f"{r['new_tokens']} greedy tokens at ctx {P}..{P + r['new_tokens']}, {r['dtype']} weights on {r['cores']} threads "
                                              f"(affinity {r['threads']['affinity']}, cgroup quota {r['threads']['cgroup_quota']}); decode tokens/s between first and last new token"}
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dump)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
