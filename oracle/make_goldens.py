"""Generate tests/golden/*.npz by running the REFERENCE's own code (imported from /root/reference) in this container.

TEST INFRASTRUCTURE ONLY -- run once by hand (`python oracle/make_goldens.py`); the resulting fixtures are committed
and are what the `-m "not gpu"` tests pin oracle/ against.  /root/reference does not exist on the GPU box, so nothing
at test/bench time imports it.

What is pinned:
  lm_tiny.npz      reference `slamkit.model.unit_lm.UnitLM` (-> HF Qwen2ForCausalLM, sdpa) forward + `compute_loss`
                   + autograd backward under bf16 autocast, then `clip_grad_norm_(0.5)` + `torch.optim.AdamW`
                   (fused) for one step, on seeded weights / tokens.  Shapes: 2 layers, hidden 128, 2 q-heads x 64,
                   1 kv-head, ffn 256, vocab 502, batch [2, 48] with right padding (labels -100).
  lm_packed.npz    the same reference model on a packed row (4 documents, restarting position_ids) with the explicit
                   block-diagonal causal 4-D mask: pins the oracle's `packed=True` path bit-exactly.
  tokeniser.npz    reference `UnitTokeniser` (load_fe=False) ids for the two example_data strings and the dedup of
                   example_data/features.jsonl (units/durations are already golden files of the reference).
  lm_loglik.npz    reference `UnitLM.log_likelihood` (sum and mean forms) on a right-padded batch, seeded weights.
  hubert_tiny.npz  reference `HubertFeatureExtractor.extract` + `batch_cluster` (HF HubertModel, sklearn
                   KMeans.predict) on seeded weights: small mHuBERT-25Hz-geometry model, 2 ragged clips.
  lm_checkpoint.npz  what the reference's `UnitLM.from_pretrained` makes of a directory written by
                   `slamkit_b200.lm.write_unit_lm_checkpoint` (seed-3 weights): its state-dict names and shapes, the
                   architecture it resolves from config.json, and its bf16 logits on seeded ids.
  audio{1,2}_head.flac  the first FLAC_HEAD_FRAMES frames of the reference's example_data/audio/audio{1,2}.flac, byte for
                   byte (libFLAC-encoded LPC streams), with the padding block dropped and STREAMINFO's sample count and
                   MD5 set to those of the kept frames; needs the built library (the decoder checks the full files first).
"""
import json
import os
import sys
import tempfile
import types

import numpy as np
import torch

REF = "/root/reference"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _stub_omegaconf():
    m = types.ModuleType("omegaconf")

    class DictConfig(dict):
        pass

    class ListConfig(list):
        pass

    class OmegaConf:
        pass

    m.DictConfig, m.ListConfig, m.OmegaConf = DictConfig, ListConfig, OmegaConf
    sys.modules["omegaconf"] = m


def bf16_to_u16(t: torch.Tensor) -> np.ndarray:
    return t.detach().contiguous().view(torch.uint16).numpy().copy()


def make_lm_golden(out_path: str):
    from oracle.lm_oracle import OracleLMConfig, init_params
    from slamkit.model.unit_lm import UnitLM, UnitLMConfig

    ocfg = OracleLMConfig(vocab_size=502, hidden=128, n_layers=2, n_heads=2, n_kv_heads=1, head_dim=64, ffn=256)
    tmp = tempfile.mkdtemp()
    json.dump({
        "architectures": ["Qwen2ForCausalLM"], "model_type": "qwen2", "hidden_size": ocfg.hidden,
        "intermediate_size": ocfg.ffn, "num_hidden_layers": ocfg.n_layers, "num_attention_heads": ocfg.n_heads,
        "num_key_value_heads": ocfg.n_kv_heads, "vocab_size": 502, "rms_norm_eps": ocfg.rms_eps,
        "max_position_embeddings": 2048, "tie_word_embeddings": True, "hidden_act": "silu",
        "rope_parameters": {"rope_theta": ocfg.rope_theta, "rope_type": "default"},
        "use_sliding_window": False, "attention_dropout": 0.0, "torch_dtype": "bfloat16",
    }, open(os.path.join(tmp, "config.json"), "w"))
    cfg = UnitLMConfig(base_model_name=tmp, vocab_size=502, twist_init=False, torch_dtype="bfloat16")
    torch.manual_seed(0)
    model = UnitLM(cfg)  # bf16 params via torch_dtype; rotary inv_freq stays fp32 as in cli/train.py
    rp = getattr(model.lm.config, "rope_parameters", None)
    assert rp and abs(rp["rope_theta"] - 10000.0) < 1e-6, rp
    params = init_params(ocfg, seed=123)
    sd = model.state_dict()
    for k, v in params.items():
        assert k in sd and sd[k].shape == v.shape, k
    missing = [k for k in sd if k not in params and k != "lm.lm_head.weight"]
    assert not missing, missing
    model.load_state_dict({**params, "lm.lm_head.weight": params["lm.model.embed_tokens.weight"]}, strict=True)
    assert model.lm.lm_head.weight.data_ptr() == model.lm.model.embed_tokens.weight.data_ptr(), "embeddings not tied"
    model.train()

    g = torch.Generator().manual_seed(7)
    B, T = 2, 48
    ids = torch.randint(2, 502, (B, T), generator=g)
    ids[:, 0] = 1
    ids[1, 40:] = 0                      # right padding as DataCollatorForLanguageModeling emits
    labels = ids.clone()
    labels[ids == 0] = -100
    attn = (ids != 0).long()
    num_items = float((labels != -100).sum())

    with torch.autocast("cpu", dtype=torch.bfloat16):
        out = model(input_ids=ids, attention_mask=attn, labels=labels, num_items_in_batch=num_items)
    loss = out.loss
    loss.backward()
    # the same batch without an attention_mask (pure causal path) and without autocast: pins the restatement bit-exactly
    with torch.no_grad():
        out_nomask = model(input_ids=ids, labels=labels, num_items_in_batch=num_items)
    grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
    logits = out.logits.detach()

    # one HF-Trainer-style optimiser step: clip 0.5 then AdamW (lr 1e-3, betas .9/.999, eps 1e-8, wd 0), fused kernel
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, fused=True)
    total_norm = torch.nn.utils.clip_grad_norm_(model.parameters(), 0.5)
    opt.step()
    new_params = {k: p.detach().clone() for k, p in model.named_parameters()}

    blob = {"ids": ids.numpy(), "labels": labels.numpy(), "num_items": np.float32(num_items),
            "loss": np.float32(loss.item()), "logits_u16": bf16_to_u16(logits),
            "loss_nomask": np.float32(out_nomask.loss.item()), "logits_nomask_u16": bf16_to_u16(out_nomask.logits),
            "total_norm": np.float32(float(total_norm)),
            "cfg": np.array([ocfg.vocab_size, ocfg.hidden, ocfg.n_layers, ocfg.n_heads, ocfg.n_kv_heads, ocfg.head_dim,
                             ocfg.ffn], dtype=np.int64)}
    for k, v in grads.items():
        blob["grad::" + k] = bf16_to_u16(v)
    for k, v in new_params.items():
        blob["new::" + k] = bf16_to_u16(v)
    np.savez_compressed(out_path, **blob)
    print("lm golden: loss", loss.item(), "total_norm", float(total_norm), "->", out_path)


def _reference_unit_lm(ocfg, seed_params: int):
    """The reference's own UnitLM (-> HF Qwen2ForCausalLM) on the oracle's seeded parameters."""
    from oracle.lm_oracle import init_params
    from slamkit.model.unit_lm import UnitLM, UnitLMConfig
    tmp = tempfile.mkdtemp()
    json.dump({
        "architectures": ["Qwen2ForCausalLM"], "model_type": "qwen2", "hidden_size": ocfg.hidden,
        "intermediate_size": ocfg.ffn, "num_hidden_layers": ocfg.n_layers, "num_attention_heads": ocfg.n_heads,
        "num_key_value_heads": ocfg.n_kv_heads, "vocab_size": ocfg.vocab_size, "rms_norm_eps": ocfg.rms_eps,
        "max_position_embeddings": 2048, "tie_word_embeddings": True, "hidden_act": "silu",
        "rope_parameters": {"rope_theta": ocfg.rope_theta, "rope_type": "default"},
        "use_sliding_window": False, "attention_dropout": 0.0, "torch_dtype": "bfloat16",
    }, open(os.path.join(tmp, "config.json"), "w"))
    cfg = UnitLMConfig(base_model_name=tmp, vocab_size=ocfg.vocab_size, twist_init=False, torch_dtype="bfloat16")
    torch.manual_seed(0)
    model = UnitLM(cfg)
    params = init_params(ocfg, seed=seed_params)
    model.load_state_dict({**params, "lm.lm_head.weight": params["lm.model.embed_tokens.weight"]}, strict=True)
    return model, params


def make_lm_packed_golden(out_path: str):
    """Packed batch (DataCollatorWithFlattening layout: one row, position_ids restarting per document).  The reference
    runs such batches through flash-attention's varlen path, which needs a GPU; the same attention pattern is given to
    the reference model here as an explicit 4-D block-diagonal causal mask (HF passes 4-D masks through unchanged), so
    the fixture is still produced by the reference's own UnitLM / HF Qwen2 code."""
    from oracle.lm_oracle import OracleLMConfig, packed_mask
    ocfg = OracleLMConfig(vocab_size=502, hidden=128, n_layers=2, n_heads=2, n_kv_heads=1, head_dim=64, ffn=256)
    model, _ = _reference_unit_lm(ocfg, 123)
    model.eval()
    g = torch.Generator().manual_seed(9)
    lens = [20, 1, 33, 42]
    docs = [torch.randint(2, 502, (n,), generator=g) for n in lens]
    ids = torch.cat(docs)[None]
    pos = torch.cat([torch.arange(n) for n in lens])[None]
    labels = ids.clone()
    for a in np.cumsum([0] + lens[:-1]):
        labels[0, a] = -100                        # DataCollatorWithFlattening: separator on each document's first token
    num_items = float((labels[:, 1:] != -100).sum())
    T = ids.shape[1]
    mask4d = torch.zeros(1, 1, T, T, dtype=torch.bfloat16).masked_fill(~packed_mask(pos), torch.finfo(torch.bfloat16).min)
    with torch.no_grad():
        out = model(input_ids=ids, attention_mask=mask4d, position_ids=pos, labels=labels, num_items_in_batch=num_items)
        alone = [model(input_ids=d[None]).logits[0] for d in docs]
    off = 0
    for n, a in zip(lens, alone):                  # each document alone == its slice of the packed row (bf16 noise)
        assert float((a.float() - out.logits[0, off:off + n].float()).abs().max()) < 2e-2
        off += n
    np.savez_compressed(out_path, ids=ids.numpy(), position_ids=pos.numpy(), labels=labels.numpy(),
                        num_items=np.float32(num_items), loss=np.float32(out.loss.item()),
                        logits_u16=bf16_to_u16(out.logits), lens=np.array(lens, dtype=np.int64),
                        cfg=np.array([ocfg.vocab_size, ocfg.hidden, ocfg.n_layers, ocfg.n_heads, ocfg.n_kv_heads,
                                      ocfg.head_dim, ocfg.ffn], dtype=np.int64))
    print("lm packed golden: loss", out.loss.item(), "->", out_path)


def make_loglik_golden(out_path: str):
    """`UnitLM.log_likelihood` (slamkit/model/unit_lm.py:184-194) of the reference model on seeded weights: a right-padded
    batch (pad id 0 is excluded from the sum), summed and mean forms.  What cli/eval.py's modelling metrics call."""
    from oracle.lm_oracle import OracleLMConfig
    ocfg = OracleLMConfig(vocab_size=502, hidden=128, n_layers=2, n_heads=2, n_kv_heads=1, head_dim=64, ffn=256)
    model, _ = _reference_unit_lm(ocfg, 3)
    model.eval()
    g = torch.Generator().manual_seed(11)
    tokens = torch.randint(2, 502, (3, 40), generator=g)
    tokens[:, 0] = 1
    tokens[1, 25:] = 0
    tokens[2, 33:] = 0
    ll_sum = model.log_likelihood(tokens.clone(), mean_nll=False)
    ll_mean = model.log_likelihood(tokens.clone(), mean_nll=True)
    np.savez_compressed(out_path, tokens=tokens.numpy(), ll_sum=ll_sum.float().numpy(), ll_mean=ll_mean.float().numpy(),
                        seed_params=np.int64(3))
    print("loglik golden:", ll_sum.tolist(), ll_mean.tolist(), "->", out_path)


def make_tokeniser_golden(out_path: str):
    from slamkit.tokeniser.unit_tokeniser import UnitTokeniser

    tok = UnitTokeniser(None, dedup=True, bos_eos_token_id=1, pad_token_id=0, num_units=500, load_fe=False)
    lines = [json.loads(l) for l in open(os.path.join(REF, "example_data", "tokens.jsonl"))]
    feats = [json.loads(l) for l in open(os.path.join(REF, "example_data", "features.jsonl"))]
    blob = {}
    for i, (ln, ft) in enumerate(zip(lines, feats)):
        enc = tok.prepare_sample(ln)
        blob[f"ids{i}"] = np.array(enc["input_ids"], dtype=np.int64)
        blob[f"units{i}"] = np.array(ft["units"], dtype=np.int64)
        blob[f"dur{i}"] = np.array(ft["duration"], dtype=np.int64)
        assert tok.stringify_representation([ft])[0] == ln["audio_repr"]
    batch = tok.string_tokenise([l["audio_repr"] for l in lines], return_tensors="pt", padding=True)
    blob["batch_ids"] = batch["input_ids"].numpy()
    blob["batch_mask"] = batch["attention_mask"].numpy()
    np.savez_compressed(out_path, **blob)
    print("tokeniser golden ->", out_path, {k: v.shape for k, v in blob.items()})


def make_hubert_golden(out_path: str):
    from sklearn.cluster import KMeans
    from transformers import HubertConfig, HubertModel
    from slamkit.feature_extractor.hubert_feature_extractor import HubertFeatureExtractor
    from oracle.hubert_oracle import OracleHubertConfig, init_hubert_params, hf_state_dict_from_oracle

    ocfg = OracleHubertConfig(conv_dim=64, hidden=128, n_heads=2, ffn=256, n_layers=3, pos_conv_kernel=16,
                              pos_conv_groups=4, n_units=50, layer=3)
    hcfg = HubertConfig(
        hidden_size=ocfg.hidden, num_hidden_layers=ocfg.n_layers, num_attention_heads=ocfg.n_heads,
        intermediate_size=ocfg.ffn, conv_dim=(ocfg.conv_dim,) * 8, conv_stride=ocfg.conv_stride,
        conv_kernel=ocfg.conv_kernel, conv_bias=False, feat_extract_norm="group", do_stable_layer_norm=False,
        num_conv_pos_embeddings=ocfg.pos_conv_kernel, num_conv_pos_embedding_groups=ocfg.pos_conv_groups,
        hidden_dropout=0.0, attention_dropout=0.0, activation_dropout=0.0, feat_proj_dropout=0.0, layerdrop=0.0,
        feat_proj_layer_norm=True, mask_time_prob=0.0, layer_norm_eps=ocfg.ln_eps)
    params = init_hubert_params(ocfg, seed=11)
    model = HubertModel(hcfg).eval()
    sd = hf_state_dict_from_oracle(params, ocfg, model.state_dict())
    model.load_state_dict(sd, strict=True)

    km = KMeans(n_clusters=ocfg.n_units, n_init=1)
    km.cluster_centers_ = params["kmeans.centers"].numpy().astype(np.float32)
    km._n_threads = 1
    km.n_features_in_ = ocfg.hidden
    km._n_features_out = ocfg.n_units

    fe = HubertFeatureExtractor.__new__(HubertFeatureExtractor)
    torch.nn.Module.__init__(fe)
    fe.layer, fe.num_units = ocfg.layer, ocfg.n_units
    fe.model, fe.config_model, fe.clustering = model, hcfg, km

    g = torch.Generator().manual_seed(5)
    S = 16000
    wav = (0.1 * torch.randn(2, S, generator=g)).clamp(-1, 1)
    lens = torch.tensor([16000, 11111])
    wav[1, 11111:] = 0
    toks = fe.extract(wav, lens)
    with torch.inference_mode():
        hs = model(torch.nn.functional.pad(wav, (40, 40)), output_hidden_states=True).hidden_states[ocfg.layer]
    blob = {"wav": wav.numpy(), "lens": lens.numpy(), "feat": hs.numpy().astype(np.float32),
            "tok0": np.asarray(toks[0], dtype=np.int64), "tok1": np.asarray(toks[1], dtype=np.int64)}
    np.savez_compressed(out_path, **blob)
    print("hubert golden ->", out_path, "frames", hs.shape, "lens", [len(t) for t in toks])


def make_checkpoint_golden(out_path: str):
    """The reference's `UnitLM.from_pretrained` on a checkpoint directory our writer produced."""
    import safetensors.torch
    from transformers import OPTConfig
    import slamkit.model.unit_lm as ref_mod
    from oracle.lm_oracle import OracleLMConfig, forward_logits, init_params
    from slamkit_b200.lm import LMConfig, write_unit_lm_checkpoint
    ocfg = OracleLMConfig(vocab_size=502, hidden=128, n_layers=2, n_heads=2, n_kv_heads=1, head_dim=64, ffn=256)
    p = init_params(ocfg, seed=3)
    tmp = tempfile.mkdtemp()
    base, ck = os.path.join(tmp, "base"), os.path.join(tmp, "ck")
    os.makedirs(base)
    write_unit_lm_checkpoint(ck, p, LMConfig(vocab_size=502, hidden=128, n_layers=2, n_heads=2, n_kv_heads=1, head_dim=64,
                                             ffn=256), base_model_name=base)
    json.dump(json.load(open(os.path.join(ck, "config.json")))["base_config"], open(os.path.join(base, "config.json"), "w"))
    # HF builds a default UnitLMConfig() to diff configs, whose base model is looked up on the hub (unit_lm.py:37,66-70)
    real = ref_mod.AutoConfig.from_pretrained
    ref_mod.AutoConfig.from_pretrained = lambda name, *a, **k: OPTConfig() if name == "facebook/opt-350M" else real(name, *a, **k)
    try:
        model = ref_mod.UnitLM.from_pretrained(ck, torch_dtype=torch.bfloat16)
    finally:
        ref_mod.AutoConfig.from_pretrained = real
    sd = model.state_dict()
    assert all(torch.equal(sd[k], p[k]) for k in p)
    assert set(safetensors.torch.load_file(os.path.join(ck, "model.safetensors"))) <= set(sd)
    g = torch.Generator().manual_seed(1)
    ids = torch.randint(2, 502, (2, 24), generator=g)
    ids[:, 0] = 1
    with torch.no_grad():
        logits = model(input_ids=ids).logits.to(torch.bfloat16)
        assert torch.equal(logits, forward_logits(p, ocfg, ids).to(torch.bfloat16))
    z = np.load(os.path.join(ROOT, "tests", "golden", "lm_loglik.npz"))
    ll = model.log_likelihood(torch.from_numpy(z["tokens"]), mean_nll=False)
    assert np.allclose(ll.float().numpy(), z["ll_sum"], rtol=1e-5, atol=1e-4)
    lc = model.lm.config
    arch = {"model_type": lc.model_type, "hidden_size": lc.hidden_size, "intermediate_size": lc.intermediate_size,
            "num_hidden_layers": lc.num_hidden_layers, "num_attention_heads": lc.num_attention_heads,
            "num_key_value_heads": lc.num_key_value_heads, "vocab_size": lc.vocab_size, "rms_norm_eps": lc.rms_norm_eps,
            "tie_word_embeddings": lc.tie_word_embeddings, "rope_theta": lc.rope_parameters["rope_theta"],
            "pad_token_id": model.config.base_config.pad_token_id}
    names = sorted(sd)
    np.savez_compressed(out_path, ids=ids.numpy(), logits_u16=bf16_to_u16(logits), names=np.array(names),
                        shapes=np.array([json.dumps(list(sd[k].shape)) for k in names]), arch=np.array(json.dumps(arch)))
    print("checkpoint golden ->", out_path, arch)


FLAC_HEAD_FRAMES = 8


def make_flac_head_golden(src: str, out_path: str, n_frames: int = FLAC_HEAD_FRAMES):
    import hashlib
    from slamkit_b200.audio_io import flac_decode_int, flac_info

    def crc8(b):
        c = 0
        for x in b:
            c ^= x
            for _ in range(8):
                c = ((c << 1) ^ 0x07) & 0xff if c & 0x80 else (c << 1) & 0xff
        return c

    info = flac_info(src)
    pcm = flac_decode_int(src)
    assert hashlib.md5(pcm.astype("<i2").tobytes()).digest() == info["md5"]      # the full decode is the encoder's audio
    d = open(src, "rb").read()
    assert d[:4] == b"fLaC"
    pos, blocks, last = 4, [], False
    while not last:
        last, kind, n = d[pos] & 0x80, d[pos] & 0x7f, int.from_bytes(d[pos + 1:pos + 4], "big")
        if kind != 1:                                                               # drop PADDING
            blocks.append(bytearray(d[pos:pos + 4 + n]))
        pos += 4 + n
    bs = int.from_bytes(blocks[0][4 + 2:4 + 4], "big")                              # fixed block size (max = min)
    assert blocks[0][0] & 0x7f == 0 and bs == int.from_bytes(blocks[0][4:6], "big") and bs == 4096
    # frame n_frames starts at the first sync code whose header (coded frame number, CRC-8) says so
    end = pos
    while True:
        end = d.index(b"\xff\xf8", end + 1)
        if d[end + 2:end + 4] == d[pos + 2:pos + 4] and d[end + 4] == n_frames and crc8(d[end:end + 5]) == d[end + 5]:
            break
    n = n_frames * bs
    si = blocks[0]
    si[4 + 13] = (si[4 + 13] & 0xf0) | ((n >> 32) & 0xf)
    si[4 + 14:4 + 18] = (n & 0xffffffff).to_bytes(4, "big")
    si[4 + 18:4 + 34] = hashlib.md5(pcm[:n].astype("<i2").tobytes()).digest()
    for b in blocks:
        b[0] &= 0x7f
    blocks[-1][0] |= 0x80
    open(out_path, "wb").write(b"fLaC" + b"".join(blocks) + d[pos:end])
    got = flac_decode_int(out_path)
    assert flac_info(out_path)["num_frames"] == n and np.array_equal(got, pcm[:n])
    print("flac head golden ->", out_path, n, "samples", os.path.getsize(out_path), "bytes")


if __name__ == "__main__":
    assert os.path.isdir(REF), "the reference is only mounted in the build container"
    _stub_omegaconf()
    sys.path.insert(0, REF)
    gd = os.path.join(ROOT, "tests", "golden")
    os.makedirs(gd, exist_ok=True)
    which = sys.argv[1:] or ["lm", "packed", "loglik", "tokeniser", "hubert", "checkpoint", "flac"]
    if "loglik" in which:
        make_loglik_golden(os.path.join(gd, "lm_loglik.npz"))
    if "lm" in which:
        make_lm_golden(os.path.join(gd, "lm_tiny.npz"))
    if "packed" in which:
        make_lm_packed_golden(os.path.join(gd, "lm_packed.npz"))
    if "tokeniser" in which:
        make_tokeniser_golden(os.path.join(gd, "tokeniser.npz"))
    if "hubert" in which:
        make_hubert_golden(os.path.join(gd, "hubert_tiny.npz"))
    if "checkpoint" in which:
        make_checkpoint_golden(os.path.join(gd, "lm_checkpoint.npz"))
    if "flac" in which:
        for name in ("audio1", "audio2"):
            make_flac_head_golden(os.path.join(REF, "example_data", "audio", f"{name}.flac"),
                                  os.path.join(gd, f"{name}_head.flac"))
