#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native slamkit hot path.

Default workload (BASELINE.json configs[1]): one optimiser step of the SLAM pre-training recipe -- Qwen2.5-0.5B-shaped
unit LM (358 M params, vocab 502, bf16 params and optimiser state), per-GPU micro-batch [8, 1024] synthetic unit
tokens, gradient clip 0.5 + AdamW -- data-parallel over N GPUs with one gradient all-reduce per step (the package's
peer-memory kernel on one node; `config.dp_comm` in the JSON line says which backend ran).

  python bench.py --gpus N --steps K --warmup W            # our arm (one JSON line on rank 0)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the reference's algorithm on the host cores
  python bench.py --workload cfg4|cfg5 ...                 # BASELINE configs[3] / [4] (see run_cfg4 / run_cfg5)

Both timed legs of the default workload go through the public trainer (`slamkit_b200.trainer.B200Trainer.train_step`, what
cli/train.py calls): token counting, global item count, forward/backward, overlapped all-reduce, clip + AdamW.

`value`  : speech-tokens/s, inputs resident in HBM, CUDA-event timed, max over ranks.
`e2e`    : same metric through the public API with HOST inputs: per step a pinned-host -> device copy of ids/labels
           and a device -> host read of the loss inside the timed region.
`roofline`: the dominant kernel (tcgen05 GEMM, ~290 launches/step) timed live with CUDA events on its launching stream
           in a separate profiling step; algorithmic FLOPs = 6 * N_matmul_params * tokens (SURVEY.md §8d).
`cpu_baseline`: oracle/lm_oracle.OracleTrainer (the pinned restatement of the reference's HF path) on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SEQ = 1024
PER_GPU_BATCH = 8
N_MATMUL_PARAMS = 24 * 14_909_440 + 502 * 896          # SURVEY.md §8d
FLOP_PER_TOKEN = 6 * N_MATMUL_PARAMS + 3 * 24 * (4 * SEQ * 896) // 2   # 2.2818 GFLOP (causal-halved attention)
GEMM_FLOP_PER_TOKEN = 6 * N_MATMUL_PARAMS


def synth_batch(rank: int, idx: int, B: int = PER_GPU_BATCH, T: int = SEQ) -> torch.Tensor:
    """SURVEY.md §8d: position 0 = BOS(1), the rest uniform in [2,501] with immediate repeats re-drawn (dedup)."""
    g = torch.Generator().manual_seed(1234 + rank + 1000 * idx)
    ids = torch.randint(2, 502, (B, T), generator=g)
    ids[:, 0] = 1
    for _ in range(4):
        rep = ids[:, 1:] == ids[:, :-1]
        if not rep.any():
            break
        fresh = torch.randint(2, 502, (B, T - 1), generator=g)
        ids[:, 1:] = torch.where(rep, fresh, ids[:, 1:])
    return ids


def usable_cpus() -> int:
    """CPU threads this process may really use: affinity mask, capped by the cgroup CPU quota (a container can see
    hundreds of host cores it is not allowed to run on; oversubscribing them makes the CPU baseline crawl)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return max(1, min(n, int(os.environ.get("SK_CPU_THREADS", "32"))))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_burst": d.get("bf16_tflops"), "bf16_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "MEASURED_PEAKS.json (of measured)"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "B200_PROFILING.md (of fallback)"}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.05)
        except Exception as e:  # NVML missing: report that instead of failing the bench
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def run_reference(args, rank: int, world: int):
    """The reference's own algorithm on the host cores (oracle port: HF Qwen2 + compute_loss + clip + AdamW restated in
    plain torch, pinned to the reference by tests/golden/lm_tiny.npz).  Rank 0 only."""
    if rank != 0:
        return
    from oracle import lm_oracle as O
    torch.set_num_threads(usable_cpus())
    cfg = O.OracleLMConfig()
    tr = O.OracleTrainer(O.init_params(cfg, seed=0), cfg, lr=1e-3, max_grad_norm=0.5)
    sample_B = 1
    batches = [synth_batch(0, i, sample_B) for i in range(2)]
    for i in range(args.warmup):
        tr.train_step(batches[i % 2], batches[i % 2].clone())
    t0 = time.perf_counter()
    for i in range(args.steps):
        tr.train_step(batches[i % 2], batches[i % 2].clone())
    dt = time.perf_counter() - t0
    tok_s = sample_B * SEQ * args.steps / dt
    line = {"impl": "reference", "metric": "speech-tokens/sec (SLAM seq=1024)", "value": tok_s, "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {**workload_config(world),
                       "reference_sample": f"each CPU step is a bounded sample of the workload: one [{sample_B},{SEQ}] micro-batch "
                                           "(not the per-GPU [8,1024]) through the same 358M model, same optimiser step"},
            "cpu_baseline": {"value": tok_s, "unit": "tokens/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"{args.steps} optimiser steps on a [{sample_B},{SEQ}] micro-batch of the same model"},
            "e2e": {"value": tok_s, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


HUBERT_B, HUBERT_S = 64, 480000                      # BASELINE.json configs[2]: batch 64 x 30 s @ 16 kHz
HUBERT_FLOP_PER_CLIP = 292.10e9                        # SURVEY.md §8d (11 layers, T=750)
HUBERT_T0 = 96015


def synth_wav(rank: int, idx: int, B: int = HUBERT_B, S: int = HUBERT_S) -> torch.Tensor:
    """SURVEY.md §8d: 0.1*randn clamped to +-1."""
    g = torch.Generator().manual_seed(4321 + rank * 1_000_000 + idx)
    return (0.1 * torch.randn(B, S, generator=g)).clamp_(-1, 1)


def run_hubert_gpu(args, rank, local_rank, world, lib, dist, outputs=None):
    """Secondary headline: HuBERT-25Hz unit extraction throughput (audio-hours/s), mHuBERT geometry, synthetic audio,
    seeded random weights; every rank extracts its own batches (no collective on this path).  `outputs` (a dict, if
    given) receives the unit ids and frame counts of the last timed batch."""
    import ctypes as C
    from slamkit_b200.feature_extractor import HubertB200Config, HubertB200FeatureExtractor, random_params
    dev = torch.device("cuda", local_rank)
    cfg = HubertB200Config()
    fe = HubertB200FeatureExtractor(cfg, random_params(cfg, seed=0), device=str(dev), max_batch=HUBERT_B,
                                    max_samples=HUBERT_S)
    host = [synth_wav(rank, i).pin_memory() for i in range(2)]
    devw = [h.to(dev) for h in host]
    n = args.steps

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def mx(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for i in range(2):
        fe.units_device(devw[i % 2], None)
    sync()
    l0 = lib.sk_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        last = fe.units_device(devw[i % 2], None)
    e1.record()
    sync()
    dev_ms = mx(e0.elapsed_time(e1))
    launches = lib.sk_launch_count() - l0
    if outputs is not None:
        outputs["hubert_units"], outputs["hubert_frames"] = (t.cpu() for t in last)
    def e2e_plain():
        for i in range(n):
            ids, nf = fe.units_device(host[i % 2], None)       # pinned host -> device inside, on the compute stream
            ids_h = ids.cpu()                                   # device -> host read of the labels (192 KB)
        return ids_h

    def e2e_prefetch():
        # what a loader with pinned memory does: batch i+1's audio crosses PCIe on a copy stream while batch i is
        # extracted; every batch is still copied from pinned host memory inside the timed region
        copy = torch.cuda.Stream(device=dev)
        cur_stream = torch.cuda.current_stream()

        def fetch(i):
            with torch.cuda.stream(copy):
                t = host[i % 2].to(dev, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
            return t, ev

        nxt = fetch(0)
        for i in range(n):
            wav_d, ev = nxt
            cur_stream.wait_event(ev)
            if i + 1 < n:
                nxt = fetch(i + 1)
            ids, nf = fe.units_device(wav_d, None)
            wav_d.record_stream(cur_stream)
            ids_h = ids.cpu()
        return ids_h

    def timed(fn):
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e2.record()
        out = fn()
        e3.record()
        sync()
        return out, mx(max(e2.elapsed_time(e3), (time.perf_counter() - t0) * 1e3))

    # ragged batch as cli/extract_features.py builds it: lengths ~ U[10 s, 30 s] sorted descending, zero tail
    gl = torch.Generator().manual_seed(99 + rank)
    lens = torch.sort(torch.randint(160000, HUBERT_S + 1, (HUBERT_B,), generator=gl), descending=True).values
    lens[0] = HUBERT_S
    ragged = devw[0].clone()
    for b in range(HUBERT_B):
        ragged[b, int(lens[b]):] = 0
    lens_d = lens.to(dev)
    fe.units_device(ragged, lens_d)
    sync()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for i in range(n):
        fe.units_device(ragged, lens_d)
    r1.record()
    sync()
    ragged_ms = mx(r0.elapsed_time(r1)) / n

    ids_h, e2e_ms = timed(e2e_plain)
    e2e_mode = "H2D on the compute stream"
    if world == 1:      # (single process only: a rank-local failure must not leave the other ranks in a barrier)
        try:
            # accepted only if it reproduces the labels of the plain loop bit for bit (same batches, deterministic kernels)
            ids_p, ms_p = timed(e2e_prefetch)
            if torch.equal(ids_p, ids_h) and ms_p < e2e_ms:
                e2e_ms, e2e_mode = ms_p, "next batch's H2D prefetched on a copy stream"
        except Exception:
            torch.cuda.synchronize()
    hours = HUBERT_B * 30.0 / 3600.0 * world
    out = {"metric": "HuBERT-25Hz unit extraction audio-hours/sec", "value": hours * n / (dev_ms / 1e3),
           "unit": "audio-hours/s", "batches": n, "ms_per_batch": dev_ms / n,
           "ragged": {"ms_per_batch": ragged_ms, "audio_hours_per_s": float(lens.sum()) / 16000.0 / 3600.0 * world / (ragged_ms / 1e3),
                      "note": "64 clips of 10-30 s (mean %.1f s) padded to 30 s: the padded frames are computed, the audio "
                              "counted is the real one" % (float(lens.float().mean()) / 16000.0)},
           "config": {"workload": "mHuBERT-25Hz geometry, 11 encoder layers + km500 argmin, batch 64 x 30 s @ 16 kHz "
                                  "synthetic audio, split-bf16 (fp32-grade) tensor-core products", "parallelism": f"dp{world}"},
           "e2e": {"value": hours * n / (e2e_ms / 1e3), "unit": "audio-hours/s",
                   "h2d_bytes_per_step": HUBERT_B * HUBERT_S * 4, "d2h_bytes_per_step": int(ids_h.numel() * 4),
                   "mode": e2e_mode},
           "gpu_launches": int(launches), "dtype": "bf16x3 (split) / fp32 accumulate"}
    if rank == 0:
        pk = peaks()
        lib.sk_prof_enable(1)
        fe.units_device(devw[0], None)
        ms = (C.c_double * 4)()
        cnt = (C.c_int64 * 4)()
        lib.sk_prof_collect(ms, cnt)
        lib.sk_prof_enable(0)
        conv0_bytes = HUBERT_B * (HUBERT_T0 * 512 * 2 * 2 + (HUBERT_S + 80) * 4)
        gbs = conv0_bytes / (ms[3] / 1e3) / 1e9 if ms[3] > 0 else None
        out["roofline"] = {"bound": "hbm", "kernel": "conv0_tc_kernel (conv0 taps + GroupNorm affine as a split-bf16 tcgen05 GEMM, "
                                                     "GELU + hi/lo split in the epilogue, channels-last TMA stores)",
                           "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                           "frac": (gbs / pk["hbm_gbs"]) if gbs else None,
                           # ncu --set full at batch 16: 3.0865 GB written + 0.0326 GB read per launch -> x4 at batch 64
                           "traffic": 4 * (3.0865e9 + 0.0326e9), "traffic_unit": "bytes/launch",
                           "traffic_source": "profiles/r02_ncu_conv0_tc.txt (batch 16, scaled x4)",
                           "algorithmic_bytes_per_launch": conv0_bytes, "peak_source": pk["source"],
                           "breakdown_ms": {"gemm": ms[0], "attention": ms[1], "conv0_apply": ms[3],
                                            "batch": dev_ms / n},
                           "tensor_tflops_fp32_equivalent": HUBERT_FLOP_PER_CLIP * HUBERT_B / (dev_ms / n / 1e3) / 1e12}
    del fe
    torch.cuda.empty_cache()
    return out


def run_hubert_reference(args):
    """CPU arm of the secondary metric: the oracle (fp32 torch restatement of the reference's HF + sklearn path)."""
    from oracle import hubert_oracle as HO
    torch.set_num_threads(usable_cpus())
    o = HO.OracleHubertConfig()
    p = HO.init_hubert_params(o, seed=0)
    wav = synth_wav(0, 0, 2, 160000)
    HO.extract(p, o, wav[:1, :32000])
    t0 = time.perf_counter()
    HO.extract(p, o, wav)
    dt = time.perf_counter() - t0
    return {"value": 2 * 10.0 / 3600.0 / dt, "unit": "audio-hours/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "one batch of 2 x 10 s clips through the fp32 oracle (HF HuBERT restatement + k-means)"}


def workload_config(world: int):
    return {"workload": "SLAM pretrain step: Qwen2.5-0.5B-shaped unit LM (358M, vocab 502), unit_hubert_25 tokens, "
                        "seq=1024, per-GPU micro-batch 8, clip 0.5 + AdamW, bf16 params/state",
            "global_batch": PER_GPU_BATCH * world, "seq_len": SEQ, "parallelism": f"dp{world}",
            "l2": "working set ~11 GB/step per GPU (activations + params + optimiser state) >> 126 MB L2"}


CFG4_VOCAB = 151_665 + 502      # Qwen2.5 tokenizer entries + 500 units + <speech>, <text> (interleaving_tokeniser.py:121-127)
CFG4_TOKENS = 8192              # packed tokens per GPU and step: documents of <= 2048 tokens in ONE row (DataCollatorWithFlattening)


DUMP_SAMPLE = 1 << 20          # elements kept of each parameter-sized buffer by --dump-outputs
DUMP_LIMIT = 64 << 20


def lm_step_outputs(model, opt, returned) -> dict:
    """What a caller of a train step holds once it returns: the step's return values, the loss statistics of its last
    forward pass, the optimiser's clip statistics, and the same seeded sample of the updated parameters, the step's
    gradients and the AdamW moments (each full buffer holds one bf16 value per parameter, 0.7 GB for the default
    workload).  Copied to the host, so later work cannot change it."""
    g = torch.Generator().manual_seed(0)
    idx = torch.randint(0, model.n_params, (min(DUMP_SAMPLE, model.n_params),), generator=g).sort().values
    idx_d = idx.to(model.device)
    out = {**returned, "lm_stats": model.stats, "optimizer_stats": opt.stats, "sample_index": idx,
           "params_sample": model.params[idx_d], "grads_sample": model.grads[idx_d],
           "exp_avg_sample": opt.exp_avg[idx_d], "exp_avg_sq_sample": opt.exp_avg_sq[idx_d]}
    return {k: torch.as_tensor(v).detach().cpu() for k, v in out.items()}


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """One DIR/<name>.npy per array: integers as float64 (exact), floating point (bf16 / fp32) as float32 (exact)."""
    import numpy as np
    conv = {}
    for name, t in arrays.items():
        t = torch.as_tensor(t).detach().cpu()
        conv[name] = (t.double() if (t.dtype == torch.float64 or not t.is_floating_point()) else t.float()).numpy()
    total = sum(a.nbytes for a in conv.values())
    assert total <= DUMP_LIMIT, f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT} byte budget"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in conv.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _timed_steps(step, n_warm, n_steps, dist, world, dev):
    """Returns (device ms, wall ms) of the n_steps timed steps and what the last of them returned."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for i in range(n_warm):
        step(i)
    barrier()
    last = None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(n_steps):
        last = step(i)
    e1.record()
    barrier()
    ms = max(e0.elapsed_time(e1), 0.0)
    wall = (time.perf_counter() - t0) * 1e3
    if world > 1:
        t = torch.tensor([ms, wall], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, wall = float(t[0]), float(t[1])
    return ms, wall, last


def run_cfg4(args, rank, local_rank, world, lib, dist):
    """BASELINE configs[3]: interleaved speech-text LM (Qwen2.5-0.5B body, text+unit vocabulary of ~152 k rows, tied 136 M
    embedding), sequences of 2048 packed into one row per step with restarting position_ids (block-diagonal attention),
    through the public trainer.  Synthetic ids uniform over the vocabulary."""
    from slamkit_b200.lm import B200UnitLM, LMConfig
    from slamkit_b200.trainer import B200Trainer
    dev = torch.device("cuda", local_rank)
    cfg = LMConfig(vocab_size=CFG4_VOCAB, max_positions=2048)
    model = B200UnitLM(cfg, device=str(dev), max_batch=1, max_seq=CFG4_TOKENS, seed=0)
    trainer = B200Trainer(model, lr=5e-4, min_lr=5e-5, warmup_steps=100, total_steps=100000, max_grad_norm=0.5)
    g = torch.Generator().manual_seed(77 + rank)
    batches = []
    for i in range(2):
        lens, left = [], CFG4_TOKENS
        while left > 0:
            n = min(left, int(torch.randint(512, 2049, (1,), generator=g)))
            lens.append(n)
            left -= n
        ids = torch.randint(0, CFG4_VOCAB, (1, CFG4_TOKENS), generator=g)
        pos = torch.cat([torch.arange(n) for n in lens])[None]
        labels = ids.clone()
        labels[pos == 0] = -100                              # separator label at every document start
        n_lab = int((labels != -100).sum())
        batches.append(({"input_ids": ids.pin_memory(), "labels": labels.pin_memory(), "position_ids": pos.pin_memory(),
                         "n_items": n_lab, "n_tokens": n_lab}, lens))
    devb = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in b.items()} for b, _ in batches]
    l0 = lib.sk_launch_count()
    ms, _, last = _timed_steps(lambda i: trainer.train_step([devb[i % 2]]), max(args.warmup, 3), args.steps, dist, world, dev)
    launches = lib.sk_launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, lm_step_outputs(model, trainer.opt, {"loss": last}))

    def e2e(i):
        b = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in batches[i % 2][0].items()}
        trainer.train_step([b])
        return trainer.last_loss()
    ms2, wall2, _ = _timed_steps(e2e, 2, args.steps, dist, world, dev)
    if rank == 0:
        n_mm = 24 * 14_909_440 + CFG4_VOCAB * 896
        attn = sum(3 * 24 * 4 * n * n * 896 // 2 for n in batches[0][1])      # causal, per document
        flop = 6 * n_mm * CFG4_TOKENS + attn
        pk = peaks()
        tps = CFG4_TOKENS * world * args.steps / (ms / 1e3)
        print(json.dumps({"metric": "speech+text tokens/sec (interleaved LM, packed seq<=2048, vocab 152167)", "value": tps,
                          "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                          "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "bf16", "data": "synthetic",
                          "config": {"workload": "cfg-4: interleaved_hubert_25 speech-text LM, Qwen2.5-0.5B body + 152167-row tied "
                                                 "embedding (494M), 8192 packed tokens per GPU and step (documents of 512-2048 "
                                                 "tokens in one row, position_ids restart), clip 0.5 + AdamW, bf16",
                                     "global_batch_tokens": CFG4_TOKENS * world, "seq_len": 2048, "parallelism": f"dp{world}",
                                     "api": "slamkit_b200.trainer.B200Trainer.train_step", "documents": batches[0][1],
                                     "l2": "working set ~20 GB/step >> 126 MB L2"},
                          "e2e": {"value": CFG4_TOKENS * world * args.steps / (max(ms2, wall2) / 1e3), "unit": "tokens/s",
                                  "h2d_bytes_per_step": 3 * CFG4_TOKENS * 8, "d2h_bytes_per_step": 4},
                          "gpu_launches": int(launches),
                          "roofline": {"bound": "tensor", "kernel": "whole step (GEMMs incl. the 152k-column lm_head, attention, CE, AdamW)",
                                       "achieved": flop / (ms / args.steps / 1e3) / 1e12, "peak": pk["bf16_sustained"],
                                       "unit": "TFLOP/s", "frac": flop / (ms / args.steps / 1e3) / 1e12 / pk["bf16_sustained"],
                                       "frac_of_burst": flop / (ms / args.steps / 1e3) / 1e12 / pk["bf16_burst"],
                                       "algorithmic_flops_per_step": flop, "traffic": None, "peak_source": pk["source"]},
                          "final_loss": trainer.reduced_loss()}), flush=True)
    else:
        trainer.reduced_loss()
    if world > 1:
        dist.destroy_process_group()


def run_cfg5(args, rank, local_rank, world, lib, dist):
    """BASELINE configs[4]: DPO step (cli/preference_alignment_train.py) on [8 chosen + 8 rejected, 1024] rows: frozen
    reference forward, policy forward, per-sequence-weighted backward, all-reduce, clip + AdamW."""
    from slamkit_b200.dpo import B200DPOTrainer
    from slamkit_b200.lm import B200UnitLM, LMConfig
    dev = torch.device("cuda", local_rank)
    pol = B200UnitLM(LMConfig(), device=str(dev), max_batch=16, max_seq=SEQ, seed=0)
    ref = B200UnitLM(LMConfig(), device=str(dev), max_batch=16, max_seq=SEQ, seed=0, trainable=False)
    tr = B200DPOTrainer(pol, ref, beta=0.1, lr=5e-5, max_grad_norm=0.5)
    host = []
    for i in range(2):
        ids = torch.cat([synth_batch(rank, 10 + i), synth_batch(rank, 20 + i)])          # [16, 1024]
        ids[8:, :256] = ids[:8, :256]                                                      # shared 256-token prompts
        labels = ids.clone()
        labels[:, :256] = -100
        host.append((ids.pin_memory(), labels.pin_memory()))
    devb = [(a.to(dev), b.to(dev)) for a, b in host]
    l0 = lib.sk_launch_count()
    ms, _, last = _timed_steps(lambda i: tr.step(*devb[i % 2]), max(args.warmup, 3), args.steps, dist, world, dev)
    launches = lib.sk_launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, lm_step_outputs(pol, tr.opt, last))
    loss_host = torch.zeros((), dtype=torch.float32).pin_memory()

    def e2e(i):
        a, b = host[i % 2]
        out = tr.step(a.to(dev, non_blocking=True), b.to(dev, non_blocking=True))
        loss_host.copy_(out["loss"], non_blocking=False)
        return float(loss_host)
    ms2, wall2, _ = _timed_steps(e2e, 2, args.steps, dist, world, dev)
    if rank == 0:
        tok = 16 * SEQ
        flop = (2 * 2 + 6) * N_MATMUL_PARAMS * tok + (2 + 3) * 24 * (4 * SEQ * 896) // 2 * tok   # ref fwd + policy fwd/bwd
        pk = peaks()
        print(json.dumps({"metric": "DPO speech-tokens/sec (8 chosen + 8 rejected rows of 1024)", "value": tok * world * args.steps / (ms / 1e3),
                          "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                          "ms_per_step": ms / args.steps, "pairs_per_s": 8 * world * args.steps / (ms / 1e3),
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                          "config": {"workload": "cfg-5: DPO step, policy + frozen reference (358M each), 8 pairs per GPU, rows of 1024 "
                                                 "(256-token shared prompt), beta 0.1, clip 0.5 + AdamW, bf16",
                                     "global_batch_pairs": 8 * world, "seq_len": SEQ, "parallelism": f"dp{world}",
                                     "api": "slamkit_b200.dpo.B200DPOTrainer.step", "l2": "working set >> 126 MB L2"},
                          "e2e": {"value": tok * world * args.steps / (max(ms2, wall2) / 1e3), "unit": "tokens/s",
                                  "h2d_bytes_per_step": 2 * tok * 8, "d2h_bytes_per_step": 4},
                          "gpu_launches": int(launches),
                          "roofline": {"bound": "tensor", "kernel": "whole step (reference forward + policy forward/backward + AdamW)",
                                       "achieved": flop / (ms / args.steps / 1e3) / 1e12, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                                       "frac": flop / (ms / args.steps / 1e3) / 1e12 / pk["bf16_sustained"],
                                       "frac_of_burst": flop / (ms / args.steps / 1e3) / 1e12 / pk["bf16_burst"],
                                       "algorithmic_flops_per_step": flop, "traffic": None, "peak_source": pk["source"]}}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg4", "cfg5"],
                    help="cfg2 (default, the headline): SLAM pretrain step; cfg4: interleaved speech-text LM, packed seq 2048, "
                         "vocab ~152k; cfg5: DPO step on [8+8, 1024] pairs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-hubert", action="store_true", help="skip the secondary HuBERT audio-hours/s measurement")
    ap.add_argument("--hubert-cpu", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them computed (rank 0) as DIR/<name>.npy: returned "
                         "loss, loss / clip statistics, a seeded sample of the parameters, gradients and AdamW moments, and "
                         "the HuBERT leg's unit ids; the inputs are the same on every run")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.hubert_cpu:
        print(json.dumps(run_hubert_reference(args)), flush=True)
        return
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from slamkit_b200 import _lib
    from slamkit_b200.lm import B200AdamW, B200UnitLM, LMConfig

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"     # keep stdout to the single JSON line (NCCL prints its version there)
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.require_cuda()

    from slamkit_b200.trainer import B200Trainer
    if args.workload == "cfg4":
        return run_cfg4(args, rank, local_rank, world, lib, dist)
    if args.workload == "cfg5":
        return run_cfg5(args, rank, local_rank, world, lib, dist)
    model = B200UnitLM(LMConfig(), device=str(dev), max_batch=PER_GPU_BATCH, max_seq=SEQ, seed=0)
    # the public trainer (what cli/train.py drives): global item count over ranks, forward/backward, bucketed all-reduce
    # overlapped with backward, clip 0.5 + AdamW, cosine schedule
    trainer = B200Trainer(model, lr=1e-3, min_lr=5e-5, warmup_steps=100, total_steps=17625, max_grad_norm=0.5,
                          overlap_comm=os.environ.get("SK_NO_OVERLAP") is None)
    NB = 4
    host = [synth_batch(rank, i).pin_memory() for i in range(NB)]
    devb = [h.to(dev) for h in host]
    counts = {"n_items": PER_GPU_BATCH * SEQ, "n_tokens": PER_GPU_BATCH * SEQ}   # labels = ids, none ignored (counted on the host)
    if os.environ.get("SK_BENCH_NO_HOSTSUM"):        # A/B switch: skip the per-step gloo sum of the counts
        counts.update({"n_items_global": PER_GPU_BATCH * SEQ * world, "n_tokens_global": PER_GPU_BATCH * SEQ * world})

    def step_device(i):
        return trainer.train_step([{"input_ids": devb[i % NB], "labels": devb[i % NB], **counts}])

    def step_e2e(i):
        # host ids in (one pinned-host -> device copy feeds input_ids and labels: a causal LM's labels ARE its ids),
        # this step's loss out (pinned D2H issued behind the backward pass; the host waits for it after the optimiser has
        # been enqueued -- what a loop that logs every step does)
        ids = host[i % NB].to(dev, non_blocking=True)
        trainer.train_step([{"input_ids": ids, "labels": ids, **counts}])
        return trainer.last_loss()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for i in range(args.warmup):
        step_device(i)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib.sk_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        last = step_device(i)
    e1.record()
    barrier()
    dev_ms = max_over_ranks(e0.elapsed_time(e1))
    launches = lib.sk_launch_count() - launches0
    outputs = lm_step_outputs(model, trainer.opt, {"loss": last}) if args.dump_outputs and rank == 0 else None

    # end-to-end through the public API with host buffers
    for i in range(2):
        step_e2e(i)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e2.record()
    trainer.reduced_loss()                      # reset the logging window
    for i in range(args.steps):
        step_e2e(i)
    e3.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max_over_ranks(max(e2.elapsed_time(e3), wall_ms))
    loss = trainer.reduced_loss()               # mean loss of the timed e2e steps, SUMMED over ranks = the global loss
    sampler.stop_flag = True
    sampler.join(timeout=2)

    tokens_per_step = PER_GPU_BATCH * SEQ * world
    value = tokens_per_step * args.steps / (dev_ms / 1e3)
    e2e_value = tokens_per_step * args.steps / (e2e_ms / 1e3)

    # live per-category device timing of one step (outside the timed regions)
    import ctypes as C
    pk = peaks()
    roof = None
    if rank == 0:
        lib.sk_prof_enable(1)
        reps = 3
        for i in range(reps):
            model.forward_backward(devb[i % NB], devb[i % NB], num_items_in_batch=float(PER_GPU_BATCH * SEQ * world))
            trainer.opt.step()
        ms = (C.c_double * 4)()
        cnt = (C.c_int64 * 4)()
        lib.sk_prof_collect(ms, cnt)
        lib.sk_prof_enable(0)
        gemm_ms, attn_ms, opt_ms = ms[0] / reps, ms[1] / reps, ms[2] / reps
        step_ms = dev_ms / args.steps
        gemm_tf = GEMM_FLOP_PER_TOKEN * PER_GPU_BATCH * SEQ / (gemm_ms / 1e3) / 1e12
        # DRAM bytes per GEMM launch (read + write), mean over the step's GEMM launches: written by tools/profile_lm_step.sh
        # from an ncu launch list of THIS build (bench.py cannot run under ncu itself)
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "r02_lm_gemm_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            traffic, traffic_src = tj["gemm_dram_bytes_per_launch"], f"profiles/r02_lm_gemm_traffic.json ({tj['source']})"
        roof = {"bound": "tensor", "kernel": f"gemm_tcgen05_kernel ({cnt[0] // reps} launches/step, fused epilogues included)",
                "achieved": gemm_tf, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                "frac": gemm_tf / pk["bf16_sustained"], "frac_of_burst": gemm_tf / pk["bf16_burst"],
                "traffic": traffic, "traffic_unit": "bytes/launch", "traffic_source": traffic_src,
                "peak_source": pk["source"] + ", sustained (frac) and burst (frac_of_burst)",
                "algorithmic_flops_per_step": GEMM_FLOP_PER_TOKEN * PER_GPU_BATCH * SEQ,
                "share_of_step": gemm_ms / step_ms,
                "breakdown_ms": {"gemm": gemm_ms, "attention": attn_ms, "optimizer": opt_ms,
                                 "other": max(step_ms - gemm_ms - attn_ms - opt_ms, 0.0), "step": step_ms},
                "step_tflops": FLOP_PER_TOKEN * PER_GPU_BATCH * SEQ / (step_ms / 1e3) / 1e12 / world * world,
                "step_frac_of_peak": FLOP_PER_TOKEN * PER_GPU_BATCH * SEQ / (step_ms / 1e3) / 1e12 / pk["bf16_sustained"],
                "step_frac_of_burst": FLOP_PER_TOKEN * PER_GPU_BATCH * SEQ / (step_ms / 1e3) / 1e12 / pk["bf16_burst"]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the CPU leg runs in a child process with a hard time box, so a slow host cannot stall the GPU result
        import subprocess
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3",
                                "--warmup", "1"], capture_output=True, text=True, timeout=420)
            ref = json.loads(r.stdout.strip().splitlines()[-1])
            cpu = ref["cpu_baseline"]
            cpu["sample"] = "3 optimiser steps on a [1,1024] micro-batch of the same 358M model (1 warm-up)"
        except Exception as e:
            cpu = {"value": None, "unit": "tokens/s", "cores": usable_cpus(), "kind": "port",
                   "sample": f"failed: {type(e).__name__}"}

    hubert = None
    if not args.skip_hubert:
        del devb
        try:
            hubert = run_hubert_gpu(args, rank, local_rank, world, lib, dist, outputs)
        except Exception as e:      # the secondary leg must never cost the primary line
            hubert = {"metric": "HuBERT-25Hz unit extraction audio-hours/sec", "value": None,
                      "error": f"{type(e).__name__}: {e}"}
        if rank == 0 and world == 1 and not args.no_cpu_baseline and hubert.get("value") is not None:
            import subprocess
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--hubert-cpu"], capture_output=True,
                                   text=True, timeout=300)
                hubert["cpu_baseline"] = json.loads(r.stdout.strip().splitlines()[-1])
            except Exception as e:
                hubert["cpu_baseline"] = {"value": None, "sample": f"failed: {type(e).__name__}"}

    if rank == 0:
        line = {"metric": "speech-tokens/sec (SLAM seq=1024)", "value": value, "unit": "tokens/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {**workload_config(world), "api": "slamkit_b200.trainer.B200Trainer.train_step",
                           "dp_comm": trainer.sync.backend},
                "clocks": sampler.summary(),
                "e2e": {"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": PER_GPU_BATCH * SEQ * 8,
                        "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / args.steps},
                "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu, "final_loss": loss,
                "secondary": hubert}
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
