"""Round-2 GPU parity tests (VERDICT r1 "next round" items 1, 5, 7, 8):
  * BASELINE configs at their TRUE widths against the CPU oracle (cfg-2: d 896, 14:2 heads, ffn 4864; cfg-3: full
    mHuBERT-25Hz geometry, 11 layers), with the exact unit-id match rate and the top-2 margin of every mismatch printed;
  * the data-parallel path on >= 2 GPUs: bucketed + overlapped all-reduce == all-gathered sum bit for bit, N-rank loss ==
    1-rank loss on the concatenated batch, DPO ranks stay identical;
  * the HF-Trainer-compatible nn.Module / autograd.Function boundary, log_likelihood against the reference fixture,
    run-to-run determinism of the whole gradient buffer, packed batches through cli/train.py, checkpoint resume.
Tolerances as tests/test_gpu_lm.py: loss 1e-3 relative, logits 8e-3, gradients 2e-2 (norm-wise), features 2e-4."""
import json
import os
import socket

import numpy as np
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _mk_lm(cfg_o, seed, max_batch, max_seq, device=DEV, trainable=True):
    from oracle import lm_oracle as O
    from slamkit_b200.lm import B200UnitLM, LMConfig
    p = O.init_params(cfg_o, seed=seed)
    cfg = LMConfig(vocab_size=cfg_o.vocab_size, hidden=cfg_o.hidden, n_layers=cfg_o.n_layers, n_heads=cfg_o.n_heads,
                   n_kv_heads=cfg_o.n_kv_heads, head_dim=cfg_o.head_dim, ffn=cfg_o.ffn, rms_eps=cfg_o.rms_eps,
                   rope_theta=cfg_o.rope_theta, tie_embeddings=cfg_o.tie_embeddings, max_positions=2048)
    m = B200UnitLM(cfg, device=device, max_batch=max_batch, max_seq=max_seq, trainable=trainable)
    m.load_hf_state_dict(p)
    return m, p


def _usable_cpus() -> int:
    """Threads for the CPU oracle: the affinity mask capped by the cgroup quota (the GPU box shows hundreds of host cores
    it may not run on; oversubscribing them makes the oracle crawl)."""
    import bench
    return bench.usable_cpus()


def _tiny_o():
    from oracle import lm_oracle as O
    return O.OracleLMConfig(vocab_size=502, hidden=128, n_layers=2, n_heads=2, n_kv_heads=1, head_dim=64, ffn=256)


# ---------------------------------------------------------------------------------------------- true-width parity (LM)
@pytest.mark.parametrize("n_layers,B,T", [(3, 2, 1024), (24, 1, 1024)])
def test_lm_true_width_vs_oracle(n_layers, B, T):
    """cfg-2 widths (Qwen2.5-0.5B body: d 896, 14 q-heads : 2 kv-heads, ffn 4864, vocab 502) at seq 1024 -- 3 layers at
    [2,1024] and all 24 layers at [1,1024] -- against the CPU oracle run twice on the same bf16 weights: in bf16 (= the
    reference's HF path, rounding for rounding) and in fp32 (the exact answer both approximate).
      * loss: within 1e-3 relative of the bf16 reference path (BASELINE north_star);
      * logits and every parameter gradient: at these widths two correct bf16 implementations differ from each other by
        their independent rounding noise (~1e-2 on the logits after a few layers), so the bar is the principled one -- the
        B200 path must be as close to the fp32 answer as the reference's own bf16 path is (factor 1.3 + a small floor)."""
    from oracle import lm_oracle as O
    torch.set_num_threads(_usable_cpus())
    cfg_o = O.OracleLMConfig(n_layers=n_layers)
    assert (cfg_o.hidden, cfg_o.n_heads, cfg_o.n_kv_heads, cfg_o.ffn, cfg_o.vocab_size) == (896, 14, 2, 4864, 502)
    m, p = _mk_lm(cfg_o, 5, B, T)
    g = torch.Generator().manual_seed(n_layers)
    ids = torch.randint(2, 502, (B, T), generator=g)
    ids[:, 0] = 1
    if B > 1:
        ids[1, 900:] = 0                      # a right-padded row
    labels = ids.clone()
    labels[ids == 0] = -100
    n_items = float((labels != -100).sum())
    ref_loss, ref_logits, ref_grads = O.forward_backward(p, cfg_o, ids, labels, n_items)
    p32 = {k: v.float() for k, v in p.items()}
    loss32, logits32, grads32 = O.forward_backward(p32, cfg_o, ids, labels, n_items)
    out = m.forward_backward(ids, labels, num_items_in_batch=n_items)
    loss = float(out.loss)
    assert abs(loss - float(ref_loss)) < 1e-3 * abs(float(ref_loss)), (loss, float(ref_loss))
    assert abs(loss - float(loss32)) < 1e-3 * abs(float(loss32)), (loss, float(loss32))
    valid = ids != 0
    ours = m.logits_view(B, T).cpu()[valid]
    e_ours, e_ref = rel_err(ours, logits32[valid]), rel_err(ref_logits[valid], logits32[valid])
    e_pair = rel_err(ours, ref_logits[valid])
    sd_g = m.state_dict_hf(grads=True)
    keys = [k for k in p if not k.endswith("k_proj.bias")]           # softmax is invariant to a key bias: true gradient 0
    g_ours = {k: rel_err(sd_g[k].cpu(), grads32[k]) for k in keys}
    g_ref = {k: rel_err(ref_grads[k], grads32[k]) for k in keys}
    worst = max(keys, key=lambda k: g_ours[k] / (g_ref[k] + 2e-3))
    print(f"true-width LM L={n_layers} [{B},{T}]: loss {loss:.6f} (bf16 ref {float(ref_loss):.6f}, fp32 {float(loss32):.6f}); "
          f"logits vs fp32: ours {e_ours:.2e}, bf16 ref {e_ref:.2e} (ours vs bf16 ref {e_pair:.2e}); worst gradient {worst}: "
          f"ours {g_ours[worst]:.2e} vs bf16 ref {g_ref[worst]:.2e}; max over tensors ours {max(g_ours.values()):.2e}, ref {max(g_ref.values()):.2e}")
    assert e_ours < 1.3 * e_ref + 1e-3, (e_ours, e_ref)
    assert e_pair < 2.0 * e_ref + 4e-3, (e_pair, e_ref)
    bad = {k: (g_ours[k], g_ref[k]) for k in keys if g_ours[k] > 1.3 * g_ref[k] + 3e-3}
    assert not bad, bad


# ---------------------------------------------------------------------------------------------- true-width parity (HuBERT)
def test_hubert_full_geometry_unit_ids_vs_oracle():
    """cfg-3 geometry (conv 512 x 8, hidden 768, 12 heads, ffn 3072, 11 layers, km500) on ragged 5-10 s clips: fp32 features
    within 2e-4, unit ids compared EXACTLY; the match rate and the fp64 top-2 margin of every mismatch are reported, and a
    mismatch is only tolerated on a near-tie (margin below the feature noise)."""
    from oracle import hubert_oracle as HO
    from test_gpu_hubert import _mk
    torch.set_num_threads(_usable_cpus())
    o = HO.OracleHubertConfig()
    assert (o.conv_dim, o.hidden, o.n_heads, o.ffn, o.layer, o.n_units) == (512, 768, 12, 3072, 11, 500)
    S = 160000
    lens = torch.tensor([160000, 131072, 96000, 80000])
    B = len(lens)
    fe, p = _mk(o, 7, B, S)
    g = torch.Generator().manual_seed(42)
    wav = (0.1 * torch.randn(B, S, generator=g)).clamp(-1, 1)
    for b in range(B):
        wav[b, lens[b]:] = 0
    want = HO.extract(p, o, wav, lens)
    got = fe.extract(wav, lens)
    assert [len(x) for x in got] == [len(x) for x in want] == [250, 205, 150, 125]
    feat = HO.features(p, o, wav)
    e_feat = rel_err(fe.features(wav).cpu(), feat)
    _, margin = HO.kmeans_margins(feat.numpy().reshape(-1, o.hidden), p["kmeans.centers"].numpy())
    margin = margin.reshape(B, -1)
    bad = [(b, int(t), float(margin[b, t])) for b in range(B) for t in np.nonzero(got[b] != want[b])[0]]
    total = sum(len(x) for x in want)
    print(f"full-geometry HuBERT: features rel err {e_feat:.2e}; unit ids exact on {total - len(bad)}/{total} frames "
          f"({100.0 * (total - len(bad)) / total:.3f} %); top-2 margins of the mismatches: {[round(m, 6) for _, _, m in bad]}")
    assert e_feat < 2e-4, e_feat
    assert all(m < 5e-3 for _, _, m in bad), bad
    assert len(bad) <= max(1, total // 500), (len(bad), total)


# ---------------------------------------------------------------------------------------------- nn.Module boundary
def test_hf_module_boundary_matches_the_core_path():
    """`B200UnitLMModule.forward(...).loss.backward()` puts the same loss / gradients in `.flat.grad` as the C-ABI call,
    state_dict speaks the reference's names, and a torch optimiser can drive it (HF Trainer's contract)."""
    from slamkit_b200.hf_module import B200UnitLMModule
    m, p = _mk_lm(_tiny_o(), 3, 2, 64)
    g = torch.Generator().manual_seed(0)
    ids = torch.randint(2, 502, (2, 64), generator=g)
    ids[:, 0] = 1
    ids[1, 50:] = 0
    labels = ids.clone()
    labels[ids == 0] = -100
    mask = (ids != 0).long()
    n = float((labels != -100).sum())
    ref = m.forward_backward(ids, labels, num_items_in_batch=n)
    ref_loss, ref_grads = float(ref.loss), m.grads.clone()
    mod = B200UnitLMModule(m)
    assert [k for k, _ in mod.named_parameters()] == ["flat"] and mod.flat.data_ptr() == m.params.data_ptr()
    out = mod(input_ids=ids, attention_mask=mask, labels=labels, num_items_in_batch=torch.tensor(n))
    assert float(out.loss) == ref_loss
    (2.0 * out.loss).backward()
    assert torch.equal(mod.flat.grad, ref_grads * 2)
    assert set(mod.state_dict()) == set(p) | {"lm.lm_head.weight"}
    with pytest.raises(ValueError):
        mod(input_ids=ids, attention_mask=mask.flip(1), labels=labels)          # left padding is refused, not ignored
    with torch.no_grad():
        ev = mod(input_ids=ids, attention_mask=mask, labels=labels, num_items_in_batch=n)   # eval: loss + logits, no gradients
    assert ev.logits.shape == (2, 64, 502) and abs(float(ev.loss) - ref_loss) < 1e-5 * abs(ref_loss)
    opt = torch.optim.AdamW(mod.parameters(), lr=1e-3, weight_decay=0.0)
    losses = []
    for _ in range(6):
        opt.zero_grad(set_to_none=True)
        o = mod(input_ids=ids, attention_mask=mask, labels=labels, num_items_in_batch=n)
        o.loss.backward()
        torch.nn.utils.clip_grad_norm_(mod.parameters(), 0.5)
        opt.step()
        losses.append(float(o.loss))
    assert losses[-1] < losses[0] - 0.05, losses


def test_log_likelihood_matches_reference_golden(golden_dir):
    """UnitLM.log_likelihood (slamkit/model/unit_lm.py:184-194) fixture produced by the reference's own class."""
    z = np.load(os.path.join(golden_dir, "lm_loglik.npz"))
    m, _ = _mk_lm(_tiny_o(), int(z["seed_params"]), 3, 40, trainable=False)
    tokens = torch.from_numpy(z["tokens"])
    ll = m.log_likelihood(tokens, mean_nll=False).float().cpu().numpy()
    lm = m.log_likelihood(tokens, mean_nll=True).float().cpu().numpy()
    assert np.allclose(ll, z["ll_sum"], rtol=4e-3, atol=0.5), (ll, z["ll_sum"])        # the fixture is bf16-rounded
    assert np.allclose(lm, z["ll_mean"], rtol=4e-3, atol=0.02), (lm, z["ll_mean"])


def test_gradient_buffer_is_bit_identical_run_to_run():
    """The whole flat gradient buffer -- including the tied embedding, whose scatter-add now runs in 64-bit fixed point."""
    m, _ = _mk_lm(_tiny_o(), 1, 4, 128)
    g = torch.Generator().manual_seed(3)
    ids = torch.randint(2, 12, (4, 128), generator=g)          # few distinct ids: heavy collisions in the embedding scatter
    ids[:, 0] = 1
    m.forward_backward(ids, ids.clone(), num_items_in_batch=512.0)
    a = m.grads.clone()
    for _ in range(3):
        m.forward_backward(ids, ids.clone(), num_items_in_batch=512.0)
        assert torch.equal(a, m.grads)
    assert float(m.tensor("embed", grad=True).float().abs().sum()) > 0


# ---------------------------------------------------------------------------------------------- trainer / CLI
def test_trainer_counts_tokens_like_the_reference_and_reports_global_loss():
    from slamkit_b200.trainer import B200Trainer
    m, _ = _mk_lm(_tiny_o(), 2, 2, 64)
    tr = B200Trainer(m, lr=1e-3, warmup_steps=0, total_steps=10, grad_accum=2, min_token_id_count=2)
    g = torch.Generator().manual_seed(0)
    mbs = []
    for k in range(2):
        ids = torch.randint(2, 502, (2, 64), generator=g)
        ids[:, 0] = 1
        ids[1, 40 + k:] = 0
        labels = ids.clone()
        labels[ids == 0] = -100
        mbs.append({"input_ids": ids, "labels": labels})
    tr.train_step(mbs)
    n_lab = sum(int((b["labels"] != -100).sum()) for b in mbs)
    assert tr.num_input_tokens_seen == n_lab - 4                      # BOS (id 1) is below min_token_id_count = 2
    loss = tr.reduced_loss()
    assert 5.5 < loss < 7.0 and tr.step_idx == 1


def _write_tokens(path, n_lines, seed):
    g = torch.Generator().manual_seed(seed)
    with open(path, "w") as f:
        for _ in range(n_lines):
            n = int(torch.randint(20, 90, (1,), generator=g))
            units = torch.randint(0, 500, (n,), generator=g).tolist()
            f.write(json.dumps({"audio_repr": "".join(f"<Un{u}>" for u in units), "file_name": "x"}) + "\n")


_TRAIN_ARGS = ["model=slam", "model.tlm_type=b200", "model.context_len=64", "model.config_args.twist_init=false",
               "+model.shape.hidden=128", "+model.shape.n_layers=2", "+model.shape.n_heads=2", "+model.shape.n_kv_heads=1",
               "+model.shape.ffn=256", "training_args.per_device_train_batch_size=4", "+training_args.logging_steps=1",
               "training_args.warmup_steps=2", "training_args.warmup_ratio=0"]


def test_cli_train_packed_batches(tmp_path):
    """`data.packing=true`: DataCollatorWithFlattening batches (one row, restarting position_ids) run through the
    block-diagonal attention kernels; the loss falls and eval / checkpoint bookkeeping follows the HF layout."""
    from cli import train
    tok = str(tmp_path / "tok.jsonl")
    _write_tokens(tok, 24, 0)
    log = train.main([f"data.train_path={tok}", f"data.val_path={tok}", "data.packing=true", *_TRAIN_ARGS,
                      "+training_args.max_steps=10", "training_args.eval_steps=5", "+training_args.save_steps=5",
                      f"training_args.output_dir={tmp_path}/run"])
    losses = [r["loss"] for r in log if "loss" in r]
    evals = [r["eval_loss"] for r in log if "eval_loss" in r]
    assert len(losses) == 10 and losses[-1] < losses[0] and len(evals) == 2 and evals[1] < evals[0]
    assert sorted(os.listdir(tmp_path / "run"))[:2] == ["checkpoint-10", "checkpoint-5"]
    st = json.load(open(tmp_path / "run" / "trainer_state.json"))
    assert st["global_step"] == 10 and st["num_input_tokens_seen"] > 0


def test_cli_train_resume_is_bit_identical(tmp_path):
    """`cont_training=true` (HF resume_from_checkpoint): 8 uninterrupted steps == the same run stopped at its step-4
    checkpoint and resumed, bit for bit (parameters, optimiser state, schedule position and data order are restored, and
    the step itself is deterministic)."""
    import shutil
    from safetensors.torch import load_file
    from cli import train
    tok = str(tmp_path / "tok.jsonl")
    _write_tokens(tok, 40, 1)
    common = [f"data.train_path={tok}", f"data.val_path={tok}", *_TRAIN_ARGS, "+training_args.save_steps=4", "+training_args.max_steps=8"]
    log_a = train.main(common + [f"training_args.output_dir={tmp_path}/a"])
    os.makedirs(tmp_path / "b")
    shutil.copytree(tmp_path / "a" / "checkpoint-4", tmp_path / "b" / "checkpoint-4")
    log_b = train.main(common + ["cont_training=true", f"training_args.output_dir={tmp_path}/b"])
    la, lb = [r for r in log_a if "loss" in r], [r for r in log_b if "loss" in r]
    assert [r["step"] for r in lb][-4:] == [5, 6, 7, 8]
    assert [r["loss"] for r in la][-4:] == [r["loss"] for r in lb][-4:]
    assert la[-1]["num_input_tokens_seen"] == lb[-1]["num_input_tokens_seen"]
    a, b = load_file(str(tmp_path / "a" / "model.safetensors")), load_file(str(tmp_path / "b" / "model.safetensors"))
    assert set(a) == set(b) and all(torch.equal(a[k], b[k]) for k in a)
    with pytest.raises(ValueError, match="No valid checkpoint"):
        train.main(common + ["cont_training=true", f"training_args.output_dir={tmp_path}/empty"])


def test_generate_on_the_cuda_path_follows_the_oracle():
    """`TokenLM.generate` (slamkit/model/token_lm.py:19-27) through the forward kernels: greedy continuation of a LEFT-padded
    batch (SpeechLM.generate's calling convention) -- every chosen token is the oracle's argmax for that prefix (up to bf16
    near-ties), the padded prompt is returned in front, `bad_words_ids` / eos / sampling arguments are honoured, and the
    nn.Module face forwards to the same code.  (The selection rules themselves are checked against transformers' own
    `generate` on CPU: tests/test_generation_cpu.py.)"""
    from oracle import lm_oracle as O
    from slamkit_b200.hf_module import B200UnitLMModule
    cfg_o = _tiny_o()
    m, p = _mk_lm(cfg_o, 5, 2, 64)
    g = torch.Generator().manual_seed(2)
    a, b = torch.randint(2, 502, (9,), generator=g), torch.randint(2, 502, (5,), generator=g)
    ids, mask = torch.zeros(2, 9, dtype=torch.long), torch.zeros(2, 9, dtype=torch.long)
    ids[0], mask[0] = a, 1
    ids[1, 4:], mask[1, 4:] = b, 1
    out = m.generate(ids, attention_mask=mask, max_new_tokens=6, do_sample=False, eos_token_id=None)
    assert out.shape == (2, 15) and torch.equal(out[:, :9], ids)
    torch.set_num_threads(_usable_cpus())
    for r, prompt in enumerate((a, b)):
        seq = prompt.tolist()
        for tok in out[r, 9:].tolist():
            lo = O.forward_logits(p, cfg_o, torch.tensor([seq]))[0, -1].float()
            assert float(lo[tok]) >= float(lo.max()) - 0.02 * float(lo.max() - lo.min()), (r, len(seq), tok, int(lo.argmax()))
            seq.append(tok)
    first = int(out[0, 9])
    out2 = m.generate(ids, attention_mask=mask, max_new_tokens=3, bad_words_ids=[[first]], eos_token_id=None)
    assert first not in out2[0, 9:].tolist()
    out3 = m.generate(ids, attention_mask=mask, max_new_tokens=4, eos_token_id=first)      # row 0 stops at once, tail = pad id
    assert int(out3[0, 9]) == first and out3[0, 10:].tolist() == [m.config.pad_token_id] * (out3.shape[1] - 10)
    torch.manual_seed(0)
    out4 = B200UnitLMModule(m).generate(ids, attention_mask=mask, max_new_tokens=5, do_sample=True, temperature=0.8, top_k=25)
    assert out4.shape[0] == 2 and 9 < out4.shape[1] <= 14 and int(out4[:, 9:].max()) < 502
    with pytest.raises(NotImplementedError):
        m.generate(ids, attention_mask=mask, num_beams=4)


# ---------------------------------------------------------------------------------------------- >= 2 GPUs
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    from oracle import lm_oracle as O
    from slamkit_b200.dpo import B200DPOTrainer
    from slamkit_b200.trainer import B200Trainer
    cfg_o = O.OracleLMConfig(vocab_size=502, hidden=128, n_layers=6, n_heads=2, n_kv_heads=1, head_dim=64, ffn=256)
    dev = f"cuda:{rank}"
    g = torch.Generator().manual_seed(7)
    full = torch.randint(2, 502, (2 * world, 96), generator=g)
    full[:, 0] = 1
    full[1, 70:] = 0
    labels = full.clone()
    labels[full == 0] = -100
    mine = slice(2 * rank, 2 * rank + 2)
    res = {}
    for overlap, comm in ((False, "nccl"), (True, "nccl"), (False, "p2p"), (True, "p2p")):
        m, _ = _mk_lm(cfg_o, 11, 2 * world, 96, device=dev)
        tr = B200Trainer(m, lr=1e-12, min_lr=0.0, warmup_steps=0, total_steps=4, overlap_comm=overlap, dp_comm=comm)   # lr ~0: weights stay put
        assert tr.sync.world == world and tr.sync.overlap == overlap
        # the peer-memory all-reduce (csrc/p2p_comm.cu) must really be the one that runs -- no silent NCCL fallback here
        assert tr.sync.backend == comm, (tr.sync.backend, comm)
        # (1) the reduced flat gradient == the sum of the all-gathered per-rank gradients, bit for bit
        n_glob = float((labels != -100).sum())
        m.forward_backward(full[mine], labels[mine], num_items_in_batch=n_glob)
        local = m.grads.clone()                     # this rank's gradients, before any reduction
        torch.cuda.synchronize()
        # the step is deterministic: the same call again, now with the reduction riding on its backward pass (in overlap
        # mode buckets are reduced IN PLACE while backward still runs, so `local` had to be taken from a separate pass)
        m.forward_backward(full[mine], labels[mine], num_items_in_batch=n_glob)
        tr.sync.reduce()
        torch.cuda.synchronize()
        gathered = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(gathered, local)
        want = gathered[0].float()
        for x in gathered[1:]:
            want = (want + x.float())
        # NCCL sums bf16 pairwise in the same order for 2 ranks; for more ranks compare within bf16 rounding of the sum
        # (the peer-memory kernel adds in rank order in fp32 and rounds once: exactly `want` for any number of ranks)
        if world == 2 or comm == "p2p":
            bad = (m.grads != want.to(torch.bfloat16)).nonzero().flatten()
            assert bad.numel() == 0, (f"overlap={overlap} comm={comm}: {bad.numel()} of {m.grads.numel()} elements differ, first {int(bad[0])}, last {int(bad[-1])}; "
                                      f"buckets {tr.sync.buckets} tail {tr.sync.tail}; max abs diff {float((m.grads.float() - want).abs().max())}")
        else:
            assert rel_err(m.grads.float().cpu(), want.cpu()) < 4e-3
        # (2) N-rank loss == 1-rank loss on the concatenated batch (HF average_tokens_across_devices semantics)
        # every rank holds the same bits after the reduction
        same = [torch.empty_like(m.grads) for _ in range(world)]
        dist.all_gather(same, m.grads)
        assert all(torch.equal(same[0], x) for x in same[1:]), f"ranks disagree after the {comm} reduction"
        for _ in range(3):                       # a few real steps: flags / epochs carry over from step to step
            tr.train_step([{"input_ids": full[mine], "labels": labels[mine]}])
        tr.sync.check()
        res[f"loss_dp_{overlap}_{comm}"] = tr.reduced_loss()
        res[f"tokens_{overlap}_{comm}"] = tr.num_input_tokens_seen
        del tr, m
    m1, _ = _mk_lm(cfg_o, 11, 2 * world, 96, device=dev)
    one = m1.forward_backward(full, labels, num_items_in_batch=float((labels != -100).sum()))
    res["loss_single"] = float(one.loss)
    res["grad_err_vs_single"] = rel_err(want.cpu(), m1.grads.float().cpu())
    # (3) DPO under data parallelism: every rank ends up with identical parameters, equal to ... a single process that saw
    # all pairs (trl DDP = mean over ranks of per-rank mean loss)
    pol, _ = _mk_lm(cfg_o, 11, 4, 48, device=dev)
    ref, _ = _mk_lm(cfg_o, 11, 4, 48, device=dev, trainable=False)
    pol.params.add_(0.01 * torch.randn(pol.params.shape, generator=torch.Generator().manual_seed(5)).to(dev).to(torch.bfloat16))
    gp = torch.Generator().manual_seed(9)
    pairs = torch.randint(2, 502, (world, 2, 2, 48), generator=gp)         # [rank, chosen/rejected, pair, T]
    pairs[..., 0] = 1
    pairs[:, 1, :, :16] = pairs[:, 0, :, :16]
    ids = torch.cat([pairs[rank, 0], pairs[rank, 1]])
    lab = ids.clone()
    lab[:, :16] = -100
    trd = B200DPOTrainer(pol, ref, beta=0.1, lr=1e-3)
    trd.step(ids, lab)
    torch.cuda.synchronize()
    allp = [torch.empty_like(pol.params) for _ in range(world)]
    dist.all_gather(allp, pol.params)
    res["dpo_ranks_identical"] = all(torch.equal(allp[0], x) for x in allp[1:])
    if rank == 0:
        json.dump(res, open(os.path.join(out_dir, "res.json"), "w"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_data_parallel_path_on_two_gpus(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_dp_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    r = json.load(open(tmp_path / "res.json"))
    print("2-GPU data-parallel check:", r)
    for key in ("False_nccl", "True_nccl", "False_p2p", "True_p2p"):
        assert abs(r[f"loss_dp_{key}"] - r["loss_single"]) < 2e-4 * abs(r["loss_single"]), r
        assert r[f"tokens_{key}"] == r["tokens_False_nccl"]
    assert r["grad_err_vs_single"] < 1e-2 and r["dpo_ranks_identical"]
