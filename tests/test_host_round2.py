"""CPU tests of the round-2 host logic: gradient-bucket plan + the product GradSync under gloo, the reference's token
counting, the packing / padding collators against HF's own, dataset mixing against `datasets`, checkpoint layout against
the reference's `UnitLM.from_pretrained`, checkpoint rotation / resume bookkeeping, rank-file merging, mask validation,
architecture validation.  No GPU: nothing here launches a kernel."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


# ------------------------------------------------------------------------------------------------ GradSync
def test_bucket_plan_covers_the_flat_buffer_exactly_once():
    from slamkit_b200.trainer import plan_buckets
    for nl, lpb in [(24, 4), (2, 4), (7, 3), (1, 1), (24, 24)]:
        sizes = [1000 + 13 * l for l in range(nl)]
        starts = [sum(sizes[:l]) for l in range(nl + 1)]
        n_params = starts[-1] + 64 + 512 * 896
        buckets, tail = plan_buckets(starts, n_params, lpb)
        cover = np.zeros(n_params, dtype=np.int32)
        for ev, lo, hi in buckets:
            assert lo == starts[ev] and lo < hi          # the bucket may go as soon as its FIRST layer's gradients are final
            cover[lo:hi] += 1
        cover[tail[0]:tail[1]] += 1
        assert (cover == 1).all()
        evs = [b[0] for b in buckets]
        assert evs == sorted(evs, reverse=True) and evs[-1] == 0     # backward order: last layers first


SYNC_WORKER = r'''
import os, sys, types, torch, torch.distributed as dist
sys.path.insert(0, os.environ["SK_ROOT"])
from slamkit_b200.trainer import GradSync, HostReducer, plan_buckets
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
nl = 5
sizes = [96 * (l + 1) for l in range(nl)]
tensors = {f"layers.{l}.ln1": (sum(sizes[:l]), 1, 8) for l in range(nl)}
tensors["final_norm"] = (sum(sizes), 1, 8)
n_params = sum(sizes) + 8 + 640
g = torch.Generator().manual_seed(100 + rank)
grads = torch.randn(n_params, generator=g)
model = types.SimpleNamespace(config=types.SimpleNamespace(n_layers=nl), tensors=tensors, n_params=n_params, grads=grads.clone(),
                              device=torch.device("cpu"))
sync = GradSync(model, layers_per_bucket=2, overlap=True)      # overlap silently off: CPU gradients
assert sync.world == 2 and not sync.overlap
assert sync.backend == "nccl" and sync.p2p is None             # host gradients: torch.distributed (here gloo), never the peer kernel
assert len(sync.buckets) == 3                                  # layers (3,4), (1,2), (0)
sync.reduce()
sync.check()
ref = grads.clone(); dist.all_reduce(ref)
assert torch.equal(model.grads, ref), float((model.grads - ref).abs().max())     # bucketed == one big all-reduce, bit for bit
tot = HostReducer().sum([3 + rank, 10.0])
assert tot == [7.0, 20.0], tot
if rank == 0: print("SYNC_OK")
'''


def test_gradsync_buckets_and_host_reducer_gloo_world2(tmp_path):
    """The PRODUCT GradSync (bucket bounds, tail) and HostReducer under a 2-rank gloo group."""
    script = tmp_path / "w.py"
    script.write_text(SYNC_WORKER)
    env = dict(os.environ, SK_ROOT=ROOT, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29641", str(script)],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "SYNC_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


def test_peer_allreduce_range_rule_and_default_bucket_size():
    """The peer-memory kernel moves 16-byte chunks: ranges must start and end on multiples of 8 bf16 elements (anything else
    goes through torch.distributed); it uses 2-layer buckets, NCCL keeps 4."""
    from slamkit_b200.p2p import MAX_SLOTS, MAX_WORLD, PeerAllReduce
    assert PeerAllReduce.supports(0, 8) and PeerAllReduce.supports(64, 64 + 896 * 8)
    assert not PeerAllReduce.supports(4, 12) and not PeerAllReduce.supports(0, 7) and not PeerAllReduce.supports(8, 8)
    assert MAX_WORLD == 8 and MAX_SLOTS >= 64
    from slamkit_b200.lm import LMConfig
    # every tensor of the LM layout starts on a 64-element boundary, so every bucket of the real model qualifies
    import types
    from slamkit_b200.trainer import plan_buckets
    cfg = LMConfig()
    per_layer = 896 + 1152 * 896 + 1152 + 896 * 896 + 896 + 9728 * 896 + 896 * 4864
    pad = lambda n: (n + 63) // 64 * 64
    starts = [l * pad(per_layer) for l in range(cfg.n_layers + 1)]
    buckets, tail = plan_buckets(starts, starts[-1] + 896 + 512 * 896, 2)
    assert len(buckets) == 12 and all(PeerAllReduce.supports(lo, hi) for _, lo, hi in buckets) and PeerAllReduce.supports(*tail)


# ------------------------------------------------------------------------------------------------ token counting
def test_count_tokens_is_the_reference_rule():
    """SLAMTrainer.get_num_tokens (slamkit/trainer/slam_trainer.py:59-66): un-shifted labels != -100, optional id range."""
    from slamkit_b200.trainer import count_tokens
    labels = torch.tensor([[1, 5, 9, 501, -100, -100], [1, 2, 3, 4, 5, 1]])
    assert count_tokens(labels) == 10
    assert count_tokens(labels, min_token_id_count=2) == 7
    assert count_tokens(labels, max_token_id_count=5) == 8
    assert count_tokens(labels, 2, 5) == 5


# ------------------------------------------------------------------------------------------------ collators
def test_padding_collator_known_answer_of_the_example_data():
    """SURVEY.md §8 a-7: the reference collator on example_data/tokens.jsonl gives [2,330] with 40 ignored / 620 valid."""
    from cli.train import collate, load_chunks
    from slamkit_b200.tokeniser import B200UnitTokeniser
    z = np.load(os.path.join(GOLDEN, "tokeniser.npz"), allow_pickle=True)
    seqs = [z["ids0"].tolist(), z["ids1"].tolist()]
    assert sorted(len(s) for s in seqs) == [290, 330], [k for k in z.files]
    b = collate(seqs, 0)
    assert tuple(b["input_ids"].shape) == (2, 330)
    assert int((b["labels"] == -100).sum()) == 40 and int((b["labels"] != -100).sum()) == 620
    assert torch.equal(b["labels"][b["labels"] != -100], b["input_ids"][b["labels"] != -100])


def test_flattening_collator_matches_hf():
    """cli/train.py's packed batches == transformers.DataCollatorWithFlattening (slamkit/data/hf_dataset.py:61-62)."""
    from transformers import DataCollatorWithFlattening
    from cli.train import collate_flattened
    g = torch.Generator().manual_seed(0)
    chunks = [[1] + torch.randint(2, 502, (n,), generator=g).tolist() + [1] for n in (5, 17, 1, 40)]
    ours = collate_flattened(chunks)
    hf = DataCollatorWithFlattening(return_tensors="pt")([{"input_ids": c} for c in chunks])
    for k in ("input_ids", "labels", "position_ids"):
        assert torch.equal(ours[k], hf[k]), k
    assert int((ours["labels"] == -100).sum()) == len(chunks)


def test_mix_datasets_matches_datasets_interleave():
    datasets = pytest.importorskip("datasets")
    from cli.train import mix_datasets
    sets = [[[0, i] for i in range(37)], [[1, i] for i in range(11)], [[2, i] for i in range(23)]]
    ratios = [0.2023584112, 0.5433262899, 0.2543152989]
    for strat in ("first_exhausted", "all_exhausted"):
        ref = datasets.interleave_datasets([datasets.Dataset.from_dict({"x": s}) for s in sets], probabilities=ratios, seed=0,
                                           stopping_strategy=strat)
        assert mix_datasets(sets, ratios, strat) == ref["x"], strat


# ------------------------------------------------------------------------------------------------ masks / architectures
def test_only_right_padding_masks_are_accepted():
    from slamkit_b200.lm import check_right_padded
    check_right_padded(None)
    check_right_padded(torch.ones(3, 7, dtype=torch.long))
    check_right_padded(torch.tensor([[1, 1, 1, 0, 0], [1, 1, 1, 1, 1], [1, 0, 0, 0, 0]]))
    with pytest.raises(ValueError):
        check_right_padded(torch.tensor([[0, 0, 1, 1, 1]]))                       # left padding
    with pytest.raises(ValueError):
        check_right_padded(torch.tensor([[1, 0, 1, 1, 0]]))                       # hole
    with pytest.raises(ValueError):
        check_right_padded(torch.ones(1, 1, 4, 4))                                # explicit 4-D mask


def test_unsupported_base_architectures_are_refused():
    from transformers import OPTConfig, Qwen2Config
    from slamkit_b200.lm import LMConfig
    with pytest.raises(ValueError, match="unsupported base architecture"):
        LMConfig.from_hf(OPTConfig(), vocab_size=502)                             # config/model/twist.yaml's OPT-125M
    c = LMConfig.from_hf(Qwen2Config(hidden_size=896, intermediate_size=4864, num_hidden_layers=24, num_attention_heads=14,
                                     num_key_value_heads=2, tie_word_embeddings=True), vocab_size=502)
    assert (c.hidden, c.ffn, c.n_layers, c.n_heads, c.n_kv_heads, c.qkv_bias) == (896, 4864, 24, 14, 2, True)
    with pytest.raises(ValueError, match="head_dim 64"):
        LMConfig.from_hf(Qwen2Config(hidden_size=1024, num_attention_heads=4, num_key_value_heads=4), vocab_size=502)


# ------------------------------------------------------------------------------------------------ checkpoints
def _tiny_cfg():
    from slamkit_b200.lm import LMConfig
    return LMConfig(vocab_size=502, hidden=128, n_layers=2, n_heads=2, n_kv_heads=1, head_dim=64, ffn=256)


def test_checkpoint_layout_round_trip(tmp_path):
    from oracle import lm_oracle as O
    from safetensors.torch import load_file
    from slamkit_b200.lm import write_unit_lm_checkpoint
    ocfg = O.OracleLMConfig(vocab_size=502, hidden=128, n_layers=2, n_heads=2, n_kv_heads=1, head_dim=64, ffn=256)
    p = O.init_params(ocfg, seed=3)
    write_unit_lm_checkpoint(str(tmp_path), p, _tiny_cfg(), base_model_name="Qwen/Qwen2.5-0.5B")
    sd = load_file(str(tmp_path / "model.safetensors"))
    assert set(sd) == set(p) and all(torch.equal(sd[k], p[k]) for k in p)
    c = json.load(open(tmp_path / "config.json"))
    assert c["model_type"] == "speech_language_model" and c["base_config"]["model_type"] == "qwen2"
    assert c["base_config"]["num_key_value_heads"] == 1 and c["vocab_size"] == 502 and c["twist_init"] is False


def test_reference_unit_lm_loads_a_b200_checkpoint(tmp_path):
    """SURVEY.md §8 f-4: the reference's own `UnitLM.from_pretrained` consumes the directory `save_pretrained` writes.
    tests/golden/lm_checkpoint.npz holds what it made of such a directory (oracle/make_goldens.py): the parameter names
    and shapes it loaded, the architecture it read from config.json, and its logits.  The directory written now must
    give the same names, shapes and architecture, and the model it describes (run by the oracle) the reference's logits
    and, under the reference's log_likelihood rule (unit_lm.py:184-194, calc_nll), its tests/golden/lm_loglik.npz."""
    from helpers import u16_to_bf16
    from oracle import lm_oracle as O
    from safetensors.torch import load_file
    from slamkit_b200.lm import write_unit_lm_checkpoint
    p = O.init_params(O.OracleLMConfig(vocab_size=502, hidden=128, n_layers=2, n_heads=2, n_kv_heads=1, head_dim=64,
                                       ffn=256), seed=3)
    write_unit_lm_checkpoint(str(tmp_path), p, _tiny_cfg(), base_model_name="Qwen/Qwen2.5-0.5B")
    z = np.load(os.path.join(GOLDEN, "lm_checkpoint.npz"))
    ref_shapes = {str(k): tuple(json.loads(str(s))) for k, s in zip(z["names"], z["shapes"])}
    sd = load_file(str(tmp_path / "model.safetensors"))
    assert {k: tuple(v.shape) for k, v in sd.items()} == {k: s for k, s in ref_shapes.items() if k != "lm.lm_head.weight"}
    assert "lm.lm_head.weight" in ref_shapes                                       # the reference ties it to the embedding
    assert all(torch.equal(sd[k], p[k]) for k in p), [k for k in p if not torch.equal(sd[k], p[k])][:3]
    base = json.load(open(tmp_path / "config.json"))["base_config"]
    arch = json.loads(str(z["arch"]))
    assert {k: base[k] for k in arch} == arch
    assert base["tie_word_embeddings"] and base["hidden_size"] // base["num_attention_heads"] == 64
    ocfg = O.OracleLMConfig(vocab_size=base["vocab_size"], hidden=base["hidden_size"], n_layers=base["num_hidden_layers"],
                            n_heads=base["num_attention_heads"], n_kv_heads=base["num_key_value_heads"], head_dim=64,
                            ffn=base["intermediate_size"], rms_eps=base["rms_norm_eps"], rope_theta=base["rope_theta"])
    with torch.no_grad():
        logits = O.forward_logits(sd, ocfg, torch.from_numpy(z["ids"]))
    assert torch.equal(logits.to(torch.bfloat16), u16_to_bf16(z["logits_u16"]))
    zl = np.load(os.path.join(GOLDEN, "lm_loglik.npz"))
    tokens = torch.from_numpy(zl["tokens"])
    with torch.no_grad():
        logits = O.forward_logits(sd, ocfg, tokens)
    target = tokens[:, 1:].clone()
    target[target == base["pad_token_id"]] = -100
    nll = torch.nn.functional.cross_entropy(logits[:, :-1].reshape(-1, logits.shape[-1]), target.reshape(-1),
                                            reduction="none").view(target.shape)
    ll = -(nll * target.ne(-100)).sum(-1)
    assert np.allclose(ll.float().numpy(), zl["ll_sum"], rtol=1e-5, atol=1e-4)


def test_checkpoint_rotation_and_listing(tmp_path):
    from cli.train import list_checkpoints, save_checkpoint
    model = types.SimpleNamespace(save_pretrained=lambda d, base_model_name=None: open(os.path.join(d, "model.safetensors"), "w").close())
    tok = types.SimpleNamespace(save_pretrained=lambda d: None)
    st = {"exp_avg": torch.zeros(8), "exp_avg_sq": torch.ones(8), "opt_step_count": 0, "num_input_tokens_seen": 0, "step_idx": 0}
    trainer = types.SimpleNamespace(state_dict=lambda: st)
    for step in (3, 6, 9, 12):
        st["opt_step_count"] = st["step_idx"] = step
        st["num_input_tokens_seen"] = 100 * step
        save_checkpoint(str(tmp_path), step, model, tok, trainer, {"cursor": 16 * step, "log_history": [], "base_model_name": "x"}, save_total_limit=2)
    ck = list_checkpoints(str(tmp_path))
    assert [os.path.basename(c) for c in ck] == ["checkpoint-9", "checkpoint-12"]     # HF save_total_limit: oldest dropped
    s = json.load(open(os.path.join(ck[-1], "trainer_state.json")))
    assert (s["global_step"], s["cursor"], s["num_input_tokens_seen"]) == (12, 192, 1200)
    o = torch.load(os.path.join(ck[-1], "optimizer.pt"))
    assert o["opt_step_count"] == 12 and torch.equal(o["exp_avg_sq"], torch.ones(8))


def test_rank_files_merge_in_global_batch_order(tmp_path):
    from cli.extract_features import merge_rank_files
    out = str(tmp_path / "f.jsonl")
    batches = [[f"b{b}_{i}" for i in range(n)] for b, n in enumerate([3, 3, 3, 3, 2])]     # 5 batches over 2 ranks
    for r in range(2):
        mine = [b for bi, b in enumerate(batches) if bi % 2 == r]
        with open(f"{out}.rank{r}", "w") as f:
            for b in mine:
                for name in b:
                    f.write(json.dumps({"file_name": name}) + "\n")
        json.dump([len(b) for b in mine], open(f"{out}.rank{r}.batches", "w"))
    merge_rank_files(out, 2)
    got = [json.loads(l)["file_name"] for l in open(out)]
    assert got == [n for b in batches for n in b]
    assert not os.path.exists(out + ".rank0") and not os.path.exists(out + ".rank1.batches")


def test_interleaving_tokeniser_on_a_local_text_tokeniser(tmp_path):
    """config/tokeniser/interleaved_hubert_25.yaml surface: an HF text tokenizer + `<Un i>`, `<speech>`, `<text>`."""
    from tokenizers import Tokenizer, models, pre_tokenizers
    from transformers import PreTrainedTokenizerFast
    from slamkit_b200.tokeniser import B200InterleavingTokeniser
    vocab = {"<pad>": 0, "<s>": 1, "hello": 2, "world": 3, "<unk>": 4}
    tk = Tokenizer(models.WordLevel(vocab, unk_token="<unk>"))
    tk.pre_tokenizer = pre_tokenizers.WhitespaceSplit()
    PreTrainedTokenizerFast(tokenizer_object=tk, unk_token="<unk>", pad_token="<pad>", bos_token="<s>").save_pretrained(str(tmp_path))
    it = B200InterleavingTokeniser(None, num_units=500, load_fe=False, text_tokeniser_path=str(tmp_path))
    assert len(it) == 5 + 500 + 2                                                  # text + units + <speech>/<text>
    ids = it.prepare_sample({"audio_repr": "<text>hello world<speech><Un3><Un499>"})["input_ids"]
    un0 = it.text_tokeniser.convert_tokens_to_ids("<Un0>")
    assert ids[-2:] == [un0 + 3, un0 + 499] and it.text_tokeniser.convert_tokens_to_ids("<speech>") == un0 + 500
    with pytest.raises(NotImplementedError):
        it.stringify_representation([{"units": [1]}], mode="train")
