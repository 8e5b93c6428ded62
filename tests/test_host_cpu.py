"""CPU-only checks of the host side: the C-ABI library loads and exports every declared symbol (no compute call), the
tokeniser mirror reproduces the reference's golden ids/strings, the compute paths fail loudly without a GPU, and the
data-parallel plumbing (one gradient all-reduce, HF num_items semantics) works over gloo with world_size 2."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    from slamkit_b200 import _lib
    lib = _lib.load()
    names = _lib.declared_symbols()
    assert len(names) > 40
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    assert lib.sk_version() >= 1


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU box")
    from slamkit_b200 import _lib, ops
    with pytest.raises(_lib.SkError):
        ops.gemm(torch.zeros(8, 8, dtype=torch.bfloat16), torch.zeros(8, 8, dtype=torch.bfloat16))
    from slamkit_b200.lm import B200UnitLM, LMConfig
    with pytest.raises(_lib.SkError):
        B200UnitLM(LMConfig(n_layers=1))


def test_product_code_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "slamkit_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dp, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "oracle/" not in src.replace("oracle/hubert_oracle.init_hubert_params", ""), f


def test_tokeniser_mirror_matches_reference_goldens(golden_dir):
    from slamkit_b200.tokeniser import B200UnitTokeniser
    z = np.load(os.path.join(golden_dir, "tokeniser.npz"))
    tok = B200UnitTokeniser(None, load_fe=False)
    assert len(tok) == 502
    strs = []
    for i in range(2):
        rep = {"units": z[f"units{i}"].tolist(), "duration": z[f"dur{i}"].tolist()}
        s = tok.stringify_representation([rep])[0]
        strs.append(s)
        assert tok.prepare_sample({"audio_repr": s})["input_ids"] == z[f"ids{i}"].tolist()
        assert tok(rep)["input_ids"] == z[f"ids{i}"].tolist()
    batch = tok.string_tokenise(strs, return_tensors="pt", padding=True)
    assert np.array_equal(batch["input_ids"].numpy(), z["batch_ids"])
    assert np.array_equal(batch["attention_mask"].numpy(), z["batch_mask"])
    dec = tok.decode_sample(batch["input_ids"][1])
    assert dec.tolist() == z["units1"].tolist()


def test_tokeniser_save_load_roundtrip(tmp_path):
    from slamkit_b200.tokeniser import B200UnitTokeniser
    B200UnitTokeniser(None, load_fe=False, num_units=500).save_pretrained(str(tmp_path))
    cfg = json.load(open(tmp_path / "tokeniser_config.json"))
    assert cfg == {"dedup": True, "bos_eos_token_id": 1, "pad_token_id": 0, "num_units": 500, "load_fe": False}
    assert len(B200UnitTokeniser.from_pretrained(str(tmp_path))) == 502


def test_hubert_weight_preparation_is_a_pure_relayout():
    """prepare_weights only permutes / pads / folds weight-norm: re-deriving the conv from the prepared matrices gives
    the oracle's fp32 result (checks the im2col ordering and the grouped positional-conv padding on CPU)."""
    from oracle import hubert_oracle as HO
    from slamkit_b200.feature_extractor import HubertB200Config, prepare_weights, GROUP_PAD
    o = HO.OracleHubertConfig(conv_dim=64, hidden=128, n_heads=2, ffn=256, n_layers=2, pos_conv_kernel=16,
                              pos_conv_groups=4, n_units=50, layer=2)
    c = HubertB200Config(conv_dim=64, hidden=128, n_heads=2, ffn=256, layer=2, pos_conv_kernel=16, pos_conv_groups=4, n_units=50)
    p = HO.init_hubert_params(o, seed=3)
    w = prepare_weights(p, c)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 64, 41, generator=g)                       # [B, C, T]
    ref = torch.nn.functional.conv1d(x, p["conv1.weight"], stride=2)
    xt = x.transpose(1, 2).contiguous()                            # channels-last
    T_out = ref.shape[-1]
    rows = torch.stack([xt[:, 2 * t:2 * t + 3].reshape(2, -1) for t in range(T_out)], 1)   # window = contiguous span
    got = rows @ w["conv1.w"].t()
    assert float((got.transpose(1, 2) - ref).abs().max()) < 1e-4
    # grouped positional conv through the padded layout
    h = torch.randn(2, 30, 128, generator=g)
    refp = torch.nn.functional.conv1d(h.transpose(1, 2), HO.pos_conv_weight(p), p["pos.bias"], padding=8, groups=4)[:, :, :-1]
    G, cg, K = 4, 32, 16
    hp = torch.zeros(2, 30 + 16, G, GROUP_PAD)
    hp[:, 8:38, :, :cg] = h.view(2, 30, G, cg)
    out = torch.zeros(2, 30, G, GROUP_PAD)
    wp = w["pos.w"].view(G, GROUP_PAD, K, GROUP_PAD)
    for t in range(30):
        win = hp[:, t:t + K]                                        # [B, K, G, 64]
        out[:, t] = torch.einsum("bkgc,gokc->bgo", win, wp) + w["pos.b"].view(G, GROUP_PAD)
    got = out[..., :cg].reshape(2, 30, 128).transpose(1, 2)
    assert float((got - refp).abs().max()) < 1e-4
    assert float(out[..., cg:].abs().max()) == 0.0


DDP_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["SK_ROOT"])
from oracle import lm_oracle as O
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
cfg = O.OracleLMConfig(vocab_size=502, hidden=64, n_layers=1, n_heads=1, n_kv_heads=1, head_dim=64, ffn=128)
p = O.init_params(cfg, seed=0)
g = torch.Generator().manual_seed(5)
full = torch.randint(2, 502, (4, 32), generator=g); full[:, 0] = 1
full[3, 20:] = 0
labels = full.clone(); labels[full == 0] = -100
mine = slice(rank * 2, rank * 2 + 2)
# the scheme bench.py / B200 trainer use: every rank normalises by the GLOBAL item count, then all-reduce(SUM)
n_local = torch.tensor([float((labels[mine] != -100).sum())]); n_glob = n_local.clone(); dist.all_reduce(n_glob)
_, _, grads = O.forward_backward(p, cfg, full[mine], labels[mine], float(n_glob))
flat = torch.cat([grads[k].float().flatten() for k in sorted(grads)])
dist.all_reduce(flat)
_, _, gref = O.forward_backward(p, cfg, full, labels, float((labels != -100).sum()))
ref = torch.cat([gref[k].float().flatten() for k in sorted(gref)])
err = float((flat - ref).norm() / ref.norm())
assert err < 2e-2, err
if rank == 0: print("DDP_OK", err)
'''


def test_data_parallel_gradient_semantics_gloo_world2(tmp_path):
    """Two CPU ranks: per-rank gradients normalised by the global token count + one SUM all-reduce == single-process
    gradients of the concatenated batch (HF Trainer num_items_in_batch / average_tokens_across_devices semantics)."""
    script = tmp_path / "w.py"
    script.write_text(DDP_WORKER)
    env = dict(os.environ, SK_ROOT=ROOT, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29631", str(script)],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DDP_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_config_loader_matches_reference_composition():
    """The Hydra-subset loader composes the same values the reference's config tree yields (SURVEY.md §5)."""
    from slamkit_b200.config import load_config
    c = load_config("extract_features", ["data_path=/x", "out_path=/y", "tokeniser.feature_extractor_type=hubert_b200"])
    fe = c.tokeniser.feature_extractor
    assert (fe.pretrained_model, fe.layer, fe.num_units) == ("slprl/mhubert-base-25hz", 11, 500)
    assert c.tokeniser.feature_extractor_type == "hubert_b200" and c.tokeniser.params.bos_eos_token_id == 1
    assert c.batch_size == 8 and c.sample_rate == 16000
    t = load_config("train", ["model=slam", "data.train_path=a", "data.val_path=b", "+training_args.max_steps=7"])
    assert t.model.context_len == 1024 and t.model.config_args.rope_theta == 10000
    assert t.model.config_args.base_model_name == "Qwen/Qwen2.5-0.5B" and t.model.config_args.twist_init is True
    assert t.training_args.learning_rate == 1e-3 and t.training_args.lr_scheduler_kwargs == {"min_lr": 5e-5}
    assert t.training_args.max_grad_norm == 0.5 and t.training_args.per_device_train_batch_size == 8
    assert t.training_args.max_steps == 7 and t.tokeniser.params.load_fe is False and t.data.packing is False
    l9 = load_config("train", ["tokeniser=unit_hubert_l9", "data.train_path=a", "data.val_path=b"])
    assert l9.tokeniser.feature_extractor.layer == 9
    with pytest.raises(ValueError):
        load_config("train", []).data.train_path          # '???' mandatory value
    with pytest.raises(KeyError):
        load_config("train", ["training_args.not_a_key=1", "data.train_path=a", "data.val_path=b"])


def test_prepare_tokens_cli_reproduces_reference_golden(golden_dir, tmp_path):
    """features.jsonl -> tokens.jsonl through cli/prepare_tokens.py equals the reference's example_data/tokens.jsonl
    content (strings decoded back to the golden unit ids; key order file_name, audio_repr)."""
    from cli import prepare_tokens
    from slamkit_b200.tokeniser import B200UnitTokeniser
    z = np.load(os.path.join(golden_dir, "tokeniser.npz"))
    fp = tmp_path / "features.jsonl"
    with open(fp, "w") as f:
        for i in range(2):
            f.write(json.dumps({"units": z[f"units{i}"].tolist(), "duration": z[f"dur{i}"].tolist(), "file_name": f"a{i}.flac"}) + "\n")
        f.write("{not json}\n")                              # swallowed with a warning, like the reference
    out = prepare_tokens.main([f"data_path={fp}", f"out_path={tmp_path}/out"])
    lines = [json.loads(x) for x in open(out)]
    assert len(lines) == 2 and list(lines[0].keys()) == ["file_name", "audio_repr"]
    tok = B200UnitTokeniser(None, load_fe=False)
    for i, ln in enumerate(lines):
        assert tok.prepare_sample(ln)["input_ids"] == z[f"ids{i}"].tolist()


@pytest.mark.parametrize("orig,new,n", [(44100, 16000, 50001), (8000, 16000, 7777), (48000, 16000, 96000),
                                        (22050, 16000, 30000), (24000, 16000, 16001), (32000, 16000, 5)])
def test_resampler_is_bit_identical_to_torchaudio(orig, new, n):
    """cli/extract_features.py:53-54 resamples with torchaudio.functional.resample's defaults; the host restatement in
    slamkit_b200.audio_io must give the same samples (float32 taps, stride-`orig` polyphase convolution)."""
    torchaudio = pytest.importorskip("torchaudio")
    from slamkit_b200.audio_io import resample
    g = torch.Generator().manual_seed(orig + new)
    x = torch.rand(2, n, generator=g) * 2 - 1
    assert torch.equal(resample(x, orig, new), torchaudio.functional.resample(x, orig, new))
    assert resample(x, new, new) is x


def test_load_wav_resamples_then_mixes_down(tmp_path):
    """WavDataset.__getitem__ order (cli/extract_features.py:52-57): resample each channel, then the channel mean."""
    torchaudio = pytest.importorskip("torchaudio")
    import wave
    from slamkit_b200.audio_io import load_audio
    g = torch.Generator().manual_seed(0)
    pcm = torch.randint(-20000, 20000, (4410, 2), generator=g, dtype=torch.int32).to(torch.int16)
    path = str(tmp_path / "stereo44k.wav")
    with wave.open(path, "wb") as w:
        w.setnchannels(2); w.setsampwidth(2); w.setframerate(44100)
        w.writeframes(pcm.numpy().tobytes())
    got = load_audio(path, 16000)
    x = (pcm.float() / 32768.0).t().contiguous()
    want = torchaudio.functional.resample(x, 44100, 16000).mean(dim=0)
    assert got.shape == (1600,) and torch.equal(got, want)


def test_wav_io_roundtrip(tmp_path):
    from slamkit_b200.audio_io import load_wav, wav_num_frames, write_wav
    x = (0.3 * torch.randn(12345, generator=torch.Generator().manual_seed(0))).clamp(-1, 1)
    p = str(tmp_path / "a.wav")
    write_wav(p, x)
    assert wav_num_frames(p) == 12345
    y = load_wav(p)
    assert float((x - y).abs().max()) <= 1.0 / 32768 + 1e-7


@pytest.mark.parametrize("ch,mode,order,porder,mid_side", [(1, "fixed", 2, 1, False), (1, "fixed", 4, 0, False),
                                                             (2, "fixed", 1, 1, True), (2, "verbatim", 0, 0, False),
                                                             (1, "constant", 0, 0, False), (2, "fixed", 3, 2, False)])
def test_flac_decoder_roundtrip(tmp_path, ch, mode, order, porder, mid_side):
    """Host-side FLAC decoder (sk_flac_*) against streams produced by the test-only encoder: PCM bit-exact, STREAMINFO
    fields and the embedded MD5 of the decoded audio reproduced (frame CRC-8/CRC-16 are verified inside the decoder)."""
    import hashlib
    from flac_writer import write_flac
    from slamkit_b200.audio_io import flac_decode_int, flac_info, load_flac
    rng = np.random.default_rng(ch * 10 + order)
    n = 5000
    t = np.arange(n)
    pcm = np.stack([(3000 * np.sin(0.01 * (c + 1) * t) + rng.integers(-200, 200, n)).astype(np.int64) for c in range(ch)], 1)
    if mode == "constant":
        pcm[:] = 1234
    p = str(tmp_path / "a.flac")
    md5 = write_flac(p, pcm, mode=mode, order=order, porder=porder, mid_side=mid_side)
    info = flac_info(p)
    assert (info["sample_rate"], info["channels"], info["bits_per_sample"], info["num_frames"]) == (16000, ch, 16, n)
    got = flac_decode_int(p)
    assert got.shape == (n, ch) and np.array_equal(got, pcm)
    assert hashlib.md5(got.astype("<i2").tobytes()).digest() == md5 == info["md5"]
    x = load_flac(p)
    assert x.shape == (n,) and abs(float(x[7]) - pcm[7].mean() / 32768.0) < 1e-7
    # corruption is detected (CRC), not silently decoded
    raw = bytearray(open(p, "rb").read())
    raw[len(raw) // 2] ^= 0x10
    open(p, "wb").write(bytes(raw))
    from slamkit_b200._lib import SkError
    with pytest.raises(SkError):
        flac_decode_int(p)


def test_flac_decoder_on_reference_example_audio(golden_dir):
    """The first 8 frames of the reference's own example_data/audio/audio{1,2}.flac (libFLAC LPC streams with seek-table
    and Vorbis-comment blocks; oracle/make_goldens.py cut them): 8 x 4096 samples, and the PCM hashes to the MD5 in
    STREAMINFO, which is that of the same samples of the full file's MD5-verified decode."""
    import hashlib
    from slamkit_b200.audio_io import flac_decode_int, flac_info
    for name, n in (("audio1_head.flac", 32768), ("audio2_head.flac", 32768)):
        info = flac_info(os.path.join(golden_dir, name))
        pcm = flac_decode_int(os.path.join(golden_dir, name))
        assert info["num_frames"] == n and pcm.shape == (n, 1)
        assert hashlib.md5(pcm.astype("<i2").tobytes()).digest() == info["md5"]


def test_preference_alignment_cli_host_path(tmp_path):
    """Config composition and data path of cli/preference_alignment_train.py (reference: cli/preference_alignment_train.py,
    config/preference_alignment_train.yaml, slamkit/data/hf_dataset.py:127-148, slam_dpo_trainer.py:40-64)."""
    from cli.preference_alignment_train import auto_bleu, load_pairs, tokenize_pairs
    from slamkit_b200.config import load_config
    from slamkit_b200.dpo import collate_pairs
    from slamkit_b200.tokeniser import B200UnitTokeniser
    cfg = load_config("preference_alignment_train", ["data.train_path=pairs.jsonl", "data.val_path=null"])
    ta = cfg.training_args
    assert ta.learning_rate == 5e-5 and ta.beta == 0.1 and ta.max_grad_norm == 0.5 and ta.lr_scheduler_type == "cosine_with_min_lr"
    assert cfg.data.repetition_filter is True and cfg.data.auto_bleu_n == 2 and cfg.data.max_auto_bleu == 0.3
    assert cfg.tokeniser.params.load_fe is False and cfg.model.tlm_type == "twist"
    from cli.train import parse_run_time
    assert parse_run_time(cfg.run_time) == 6 * 3600        # YAML 1.1 reads 6:00:00 as the sexagesimal integer 21600
    # auto-BLEU: share of n-grams that occur more than once (calc_auto_bleu)
    assert auto_bleu("the cat the cat sat", 2) == 0.5 and auto_bleu("a b c d", 2) == 0.0 and auto_bleu("one", 2) == 0.0
    rows = [
        {"prompt": "<Un1><Un2>", "chosen": "<Un3><Un4>", "rejected": "<Un5>", "prompt_text": "he said", "chosen_text": "hello there", "extra": 1},
        {"prompt": "<Un7>", "chosen": "<Un8>", "rejected": "<Un9>", "prompt_text": "go go go go", "chosen_text": "go go go", "extra": 2},
        {"prompt": "<Un10><Un11><Un12>", "chosen": "<Un13>", "rejected": "<Un14><Un15>", "prompt_text": "a b", "chosen_text": "c d", "extra": 3},
    ]
    path = tmp_path / "pairs.jsonl"
    path.write_text("\n".join(json.dumps(r) for r in rows) + "\n")
    kept = load_pairs(str(path), True, 2, 0.3)
    assert [r["prompt"] for r in kept] == ["<Un1><Un2>", "<Un10><Un11><Un12>"] and set(kept[0]) == {"prompt", "chosen", "rejected"}
    assert len(load_pairs(str(path), False, 2, 0.3)) == 3
    tok = B200UnitTokeniser(None, dedup=True, bos_eos_token_id=1, pad_token_id=0, num_units=500, load_fe=False)
    t = tokenize_pairs(kept, tok, max_prompt_length=2, max_length=3)
    assert t[0]["prompt_input_ids"] == [3, 4] and t[1]["prompt_input_ids"] == [13, 14]    # left-truncated: the BOS drops first
    assert t[0]["chosen_input_ids"] == [5] and t[1]["rejected_input_ids"] == [16]          # room = max_length - len(prompt) = 1
    full = tokenize_pairs(kept, tok, max_prompt_length=None, max_length=None)
    assert full[0]["prompt_input_ids"] == [1, 3, 4] and full[0]["chosen_input_ids"] == [5, 6, 1] and full[0]["rejected_input_ids"] == [7, 1]
    ids, labels = collate_pairs(full[:1], 0)               # one pair -> [prompt+chosen ; prompt+rejected]
    assert ids.shape == (2, 6) and ids[0].tolist() == [1, 3, 4, 5, 6, 1] and labels[0].tolist() == [-100, -100, -100, 5, 6, 1]
    assert ids[1].tolist() == [1, 3, 4, 7, 1, 0] and labels[1].tolist() == [-100, -100, -100, 7, 1, -100]
    assert collate_pairs(full, 0)[0].shape == (4, 7)


def test_preference_feature_extractor_host_path(tmp_path):
    """cli/preference_alignment_feature_extractor.py: triplet batching order [prompts, chosens, rejecteds] and how the
    representations are split back into the rows (reference pad_collate_fn / extract_features, :50-82)."""
    from cli.preference_alignment_feature_extractor import attach, collate_triplets, read_triplets
    from slamkit_b200.audio_io import write_wav
    from slamkit_b200.config import load_config
    cfg = load_config("preference_alignment_feature_extractor", ["data_path=a.jsonl", "out_path=b.jsonl"])
    assert cfg.batch_size == 8 and cfg.sample_rate == 16000 and cfg.skip is None and cfg.tokeniser.tokeniser_type == "unit"
    rows = []
    for i in range(3):
        r = {"id": i}
        for j, k in enumerate(("prompt", "chosen", "rejected")):
            pth = str(tmp_path / f"{k}{i}.wav")
            write_wav(pth, torch.full((100 * (i + 1) + 10 * j,), 0.01 * (3 * i + j + 1)))
            r[f"{k}_path"] = pth
        rows.append(r)
    (tmp_path / "t.jsonl").write_text("\n".join(json.dumps(r) for r in rows) + "\n")
    got = read_triplets(str(tmp_path / "t.jsonl"), skip=1, take=None)
    assert [r["id"] for r in got] == [1, 2]
    wav, lens = collate_triplets(got)
    assert lens.tolist() == [200, 300, 210, 310, 220, 320] and wav.shape == (6, 320)
    assert abs(float(wav[2, 0]) - 0.05) < 1e-4 and float(wav[0, 250]) == 0.0          # chosen of row 1; zero padding
    reps = [{"units": [k], "duration": [1]} for k in range(6)]
    out = attach(got, reps)
    assert out[0]["prompt"]["units"] == [0] and out[1]["prompt"]["units"] == [1] and out[0]["chosen"]["units"] == [2]
    assert out[1]["rejected"]["units"] == [5] and json.loads(json.dumps(out[0]))["id"] == 1


def test_ctypes_call_sites_match_header_arity():
    """The Python side calls the C ABI through untyped ctypes: a changed prototype would only show up as garbage on the
    GPU.  Every `lib.sk_*(...)` call in the package, bench, tools and tests must pass exactly as many arguments as
    include/slamkit_b200.h declares."""
    import ast
    import glob
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(root, "include", "slamkit_b200.h")).read(), flags=re.S)
    protos = {}
    for m in re.finditer(r"\b(sk_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", hdr, flags=re.S):
        args = m.group(2).strip()
        protos[m.group(1)] = 0 if args in ("", "void") else len(args.split(","))
    assert len(protos) >= 60
    files = glob.glob(os.path.join(root, "slamkit_b200", "*.py")) + glob.glob(os.path.join(root, "tools", "*.py")) + \
        glob.glob(os.path.join(root, "tests", "*.py")) + [os.path.join(root, "bench.py"), os.path.join(root, "__graft_entry__.py")]
    bad, seen = [], set()
    for f in files:
        for node in ast.walk(ast.parse(open(f).read())):
            if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr in protos \
                    and not any(isinstance(a, ast.Starred) for a in node.args):
                seen.add(node.func.attr)
                if len(node.args) != protos[node.func.attr]:
                    bad.append((os.path.relpath(f, root), node.lineno, node.func.attr, len(node.args), protos[node.func.attr]))
    assert not bad, bad
    assert {"sk_lm_forward_backward", "sk_hubert_units", "sk_gemm_bf16_ws", "sk_attn_tc_bwd", "sk_seg_bounds"} <= seen
