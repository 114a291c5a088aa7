"""CPU: configuration records, checkpoint-key normalisation, synthetic checkpoints, session sharding."""
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest
import torch

from moshi_b200.config import LMConfig, MimiConfig, MOSHI_7B, tiny_lm_config
from moshi_b200.models.state_dict import normalize_lm_state_dict, normalize_mimi_state_dict
from moshi_b200.serving import shard_sessions
from moshi_b200.synth import lm_tensor_specs, seanet_layout, synth_lm_state_dict, synth_mimi_state_dict

ROOT = Path(__file__).resolve().parent.parent


def test_7b_config_matches_reference_json():
    # values of configs/moshi_7b_202409.json (SURVEY.md 8a)
    c = MOSHI_7B
    assert (c.dim, c.num_layers, c.num_heads, c.context) == (4096, 32, 32, 3000)
    assert c.ffn_hidden == 11264 and c.depformer_ffn_hidden == 2816
    assert c.max_delay == 1 and c.num_codebooks == 17
    total = sum(int(torch.tensor(shape).prod()) for _, shape, _ in lm_tensor_specs(c))
    assert abs(total / 1e9 - 7.688) < 0.01            # SURVEY.md: 7.688 B parameters


def test_lm_config_rejects_options_outside_hot_path(golden_dir):
    d = MOSHI_7B.to_reference_kwargs()
    d["depformer_causal"] = True                       # deprecated key is accepted and dropped
    LMConfig.from_dict(d)
    with pytest.raises(ValueError):
        LMConfig.from_dict({**d, "norm": "layer_norm"})
    with pytest.raises(ValueError):                    # only LUT conditioners fused by sum are on the step path
        LMConfig.from_dict({**d, "conditioners": {"speaker": {"type": "tensor", "tensor": {"dim": 512}}}})
    with pytest.raises(ValueError):
        LMConfig.from_dict({**d, "fuser": {"cross": ["description"]}})
    with pytest.raises(ValueError):                    # ADVICE r1: options that used to load silently
        LMConfig.from_dict({**d, "causal": False})
    with pytest.raises(ValueError):
        LMConfig.from_dict({**d, "depformer_context": 4})
    # the reference's configs/moshi_dev_2b.json, stored unmodified
    two_b = json.loads((golden_dir / "moshi_dev_2b.json").read_text())
    c2 = LMConfig.from_dict(two_b)                     # configs/moshi_dev_2b.json is inside the family now
    assert (c2.n_q, c2.dep_q, c2.max_delay) == (32, 16, 2) and "description" in c2.conditioners
    assert "conditioners" not in c2.to_reference_kwargs()


def test_mimi_config_roundtrip_and_layout():
    cfg = MimiConfig()
    assert cfg.frame_size == 1920 and cfg.hop_length == 960 and cfg.resample_stride == 2
    assert MimiConfig.from_reference_dict(cfg.to_reference_dict()) == cfg
    enc, dec = seanet_layout(cfg)
    assert [l[1] for l in enc if l[0] == "conv"] == [0, 3, 6, 9, 12, 14]     # SURVEY.md appendix A
    assert [l[1] for l in dec if l[0] == "convtr"] == [2, 5, 8, 11]
    for section, key, value in (("seanet", "pad_mode", "reflect"), ("seanet", "activation", "ReLU"), ("seanet", "causal", False),
                                ("seanet", "disable_norm_outer_blocks", 1), ("transformer", "causal", False),
                                ("transformer", "conv_layout", False)):
        bad = cfg.to_reference_dict()
        bad[section][key] = value
        with pytest.raises(ValueError):
            MimiConfig.from_reference_dict(bad)


def test_synth_checkpoints_have_reference_keys():
    sd = synth_mimi_state_dict(MimiConfig(), seed=1)
    assert sd["encoder.model.12.conv.conv.weight"].shape == (1024, 512, 16)
    assert sd["decoder.model.2.convtr.convtr.weight"].shape == (1024, 512, 16)
    assert sd["quantizer.rvq_rest.vq.layers.30._codebook.embedding_sum"].shape == (2048, 256)
    assert sd["upsample.convtr.convtr.convtr.weight"].shape == (512, 1, 4)
    assert len(sd) == 318
    a = synth_lm_state_dict(tiny_lm_config(), seed=7)
    b = synth_lm_state_dict(tiny_lm_config(), seed=7)
    assert all(torch.equal(a[k], b[k]) for k in a) and len(a) == len(lm_tensor_specs(tiny_lm_config()))


def test_legacy_checkpoint_names_are_normalised():
    w = torch.arange(2 * 3 * 4 * 4, dtype=torch.float32).view(2 * 12, 4)
    sd = normalize_lm_state_dict({"depformer.layers.0.self_attn.in_proj_weight": w,
                                  "depformer.layers.0.self_attn.out_proj.weight": torch.zeros(8, 4)})
    assert torch.equal(sd["depformer.layers.0.self_attn.in_projs.1.weight"], w[12:])
    assert sd["depformer.layers.0.self_attn.out_projs.1.weight"].shape == (4, 4)
    m = normalize_mimi_state_dict({"quantizer.rvq_first.vq.layers.0._codebook.embed_sum": torch.zeros(2, 2),
                                   "quantizer.rvq_first.vq.layers.0._codebook.cluster_size": torch.ones(2)})
    assert set(m) == {"quantizer.rvq_first.vq.layers.0._codebook.embedding_sum",
                      "quantizer.rvq_first.vq.layers.0._codebook.cluster_usage"}


def test_session_sharding_is_a_partition():
    for total in (1, 7, 512):
        for world in (1, 2, 4, 8):
            parts = [shard_sessions(total, world, r) for r in range(world)]
            flat = [s for p in parts for s in range(p.start, p.stop)]
            assert flat == list(range(total))
            assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1


def test_two_rank_replicas_over_gloo(tmp_path):
    """world_size 2 on CPU: each rank owns a disjoint shard of the sessions, the only exchange is the
    timing reduction bench.py performs (max over ranks) — same code path as the NCCL launch."""
    script = tmp_path / "w.py"
    script.write_text(
        "import os, sys, json, torch, torch.distributed as dist\n"
        f"sys.path.insert(0, {str(ROOT)!r})\n"
        "from moshi_b200.serving import shard_sessions, init_distributed, max_over_ranks, sum_over_ranks\n"
        "rank, world = init_distributed(backend='gloo')\n"
        "mine = shard_sessions(11, world, rank)\n"
        "t = max_over_ranks(float(rank + 1))\n"
        "n = sum_over_ranks(float(len(mine)))\n"
        "if rank == 0: print(json.dumps({'t': t, 'n': n, 'world': world}))\n"
        "dist.destroy_process_group()\n")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29517", str(script)],
                         capture_output=True, text=True, env=env, timeout=240)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line) == {"t": 2.0, "n": 11.0, "world": 2}


def test_session_pool_frames_and_slot_updates():
    """PCM framing and slot bookkeeping in front of DialogueService.step (server.py:116-126, batched_asr.py:146-170)."""
    import numpy as np

    from moshi_b200.serving import ACTIVE, NODATA, RESET, SessionPool
    pool = SessionPool(batch_size=3, frame_size=8, max_buffered_frames=4)
    a, b = pool.open(), pool.open()
    assert (a, b) == (0, 1) and pool.free_slots == 1
    pcm = np.full(3 * 8, 7.0, dtype=np.float32)
    upd = np.zeros(3, dtype=np.int32)
    pool.push_pcm(a, np.arange(11, dtype=np.float32))          # one frame and three samples
    pool.push_pcm(b, np.arange(5, dtype=np.float32))           # not a frame yet
    assert pool.next_frame(pcm, upd) == [a]
    assert list(upd) == [RESET, NODATA, NODATA]
    assert np.array_equal(pcm[:8], np.arange(8)) and not pcm[8:].any()
    pool.push_pcm(a, np.arange(100, 105, dtype=np.float32))    # 3 + 5 = the next frame
    pool.push_pcm(b, np.arange(5, 16, dtype=np.float32))       # two frames buffered for b
    assert pool.next_frame(pcm, upd) == [a, b]
    assert list(upd) == [ACTIVE, RESET, NODATA]
    assert np.array_equal(pcm[:8], [8, 9, 10, 100, 101, 102, 103, 104]) and np.array_equal(pcm[8:16], np.arange(8))
    assert pool.next_frame(pcm, upd) == [b] and list(upd) == [NODATA, ACTIVE, NODATA]
    assert pool.next_frame(pcm, upd) == [] and list(upd) == [NODATA] * 3
    pool.close(a)
    c = pool.open()                                            # the freed slot is handed out again and starts with RESET
    assert c == a
    pool.push_pcm(c, np.zeros(8, dtype=np.float32))
    assert pool.next_frame(pcm, upd) == [c] and upd[c] == RESET
    with pytest.raises(KeyError):
        pool.push_pcm(2, np.zeros(4, dtype=np.float32))
    with pytest.raises(OverflowError):
        pool.push_pcm(b, np.zeros(33, dtype=np.float32))
    pool.open()
    with pytest.raises(RuntimeError):
        pool.open()


def test_candle_layout_checkpoint_maps_back_to_reference_names():
    """``scripts/import_rust.py:45-113`` writes the layout ``rust/moshi-core`` loads (per-step depformer slices); restated here
    on the synthetic checkpoint and mapped back by ``normalize_lm_state_dict``: every tensor returns under its reference name."""
    import torch
    from moshi_b200.models.state_dict import normalize_lm_state_dict
    cfg = tiny_lm_config()
    sd = synth_lm_state_dict(cfg, seed=3)
    # the reference-side packed names first (what the .pt checkpoints import_rust.py reads carry)
    packed = {}
    for layer in range(cfg.depformer_num_layers):
        p = f"depformer.layers.{layer}.self_attn."
        packed[p + "in_proj_weight"] = torch.cat([sd[p + f"in_projs.{k}.weight"] for k in range(cfg.dep_q)])
        packed[p + "out_proj.weight"] = torch.cat([sd[p + f"out_projs.{k}.weight"] for k in range(cfg.dep_q)])
    candle = {k: v for k, v in sd.items() if k.startswith(("text_emb", "text_linear", "out_norm", "emb.", "transformer."))}
    for k in range(cfg.dep_q):
        base = f"depformer.{k}."
        candle[base + "linear_in.weight"] = sd[f"depformer_in.{k}.weight"]
        candle[base + "linear_out.weight"] = sd[f"linears.{k}.weight"]
        candle[base + "emb.weight"] = sd["depformer_text_emb.weight"] if k == 0 else sd[f"depformer_emb.{k - 1}.weight"]
        for layer in range(cfg.depformer_num_layers):
            src, dst = f"depformer.layers.{layer}.", base + f"transformer.layers.{layer}."
            candle[dst + "self_attn.in_proj_weight"] = packed[src + "self_attn.in_proj_weight"].chunk(cfg.dep_q)[k]
            candle[dst + "self_attn.out_proj.weight"] = packed[src + "self_attn.out_proj.weight"].chunk(cfg.dep_q)[k]
            candle[dst + "norm1.alpha"] = sd[src + "norm1.alpha"]
            candle[dst + "norm2.alpha"] = sd[src + "norm2.alpha"]
            candle[dst + "gating.linear_in.weight"] = sd[src + f"gating.{k}.linear_in.weight"]
            candle[dst + "gating.linear_out.weight"] = sd[src + f"gating.{k}.linear_out.weight"]
    back = normalize_lm_state_dict(candle)
    assert set(back) == set(sd), set(back) ^ set(sd)
    assert all(torch.equal(back[k], sd[k]) for k in sd)
    # tensor by tensor, the way LMModel streams a checkpoint in
    one = normalize_lm_state_dict({"depformer.3.transformer.layers.1.gating.linear_out.weight": candle["depformer.3.transformer.layers.1.gating.linear_out.weight"]})
    assert list(one) == ["depformer.layers.1.gating.3.linear_out.weight"]
