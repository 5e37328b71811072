"""stylesinger_b200/formats.py against the reference's own writers / loaders (their outputs on the inputs below are stored
in tests/golden/ref_formats.npz by tools/make_golden.py formats) and against hand-written files."""
import json
import os
import pickle

import numpy as np
import pytest
import torch

from stylesinger_b200 import formats as F
from tests.common import GOLDEN


def _ref():
    return np.load(os.path.join(GOLDEN, "ref_formats.npz"))


def _tiny_sd(seed):
    g = torch.Generator().manual_seed(seed)
    return {"encoder.w": torch.randn(3, 4, generator=g), "encoder.b": torch.randn(3, generator=g),
            "postdiff.denoise_fn.x": torch.randn(2, 2, generator=g)}


def test_checkpoint_selection_and_key_layouts(tmp_path):
    d = str(tmp_path)
    torch.save({"state_dict": {"model": _tiny_sd(1)}}, os.path.join(d, "model_ckpt_steps_2000.ckpt"))
    torch.save({"state_dict": {"model": _tiny_sd(2)}}, os.path.join(d, "model_ckpt_steps_160000.ckpt"))
    torch.save({"state_dict": {"model": _tiny_sd(3)}}, os.path.join(d, "model_ckpt_steps_90000.ckpt"))
    assert [os.path.basename(p) for p in F.list_checkpoints(d)] == ["model_ckpt_steps_160000.ckpt", "model_ckpt_steps_90000.ckpt",
                                                                    "model_ckpt_steps_2000.ckpt"]
    sd, path = F.load_state_dict(d)
    assert path.endswith("160000.ckpt") and all(torch.equal(sd[k], v) for k, v in _tiny_sd(2).items())
    sd, _ = F.load_state_dict(os.path.join(d, "model_ckpt_steps_2000.ckpt"))  # explicit file
    assert torch.equal(sd["encoder.w"], _tiny_sd(1)["encoder.w"])
    # flat layout ('model.' prefix) and a dotted model name (sub-module of a nested dict)
    flat = os.path.join(d, "flat.ckpt")
    torch.save({"state_dict": {"model." + k: v for k, v in _tiny_sd(4).items()}}, flat)
    sd, _ = F.load_state_dict(flat)
    assert sorted(sd) == sorted(_tiny_sd(4)) and torch.equal(sd["encoder.b"], _tiny_sd(4)["encoder.b"])
    sd, _ = F.load_state_dict(os.path.join(d, "model_ckpt_steps_2000.ckpt"), "model.encoder")
    assert sorted(sd) == ["b", "w"]
    with pytest.raises(FileNotFoundError):
        F.load_state_dict(str(tmp_path / "empty_dir_that_does_not_exist"))


def test_checkpoint_loader_agrees_with_the_reference_load_ckpt(tmp_path):
    """Two checkpoints of a small module in one work dir: the state dict the reference's load_ckpt put into the module
    (it picks the newest step) is what F.load_state_dict returns."""
    g = _ref()
    d = str(tmp_path)
    for step in (7, 3):
        sd = {k[len(f"ckpt{step}_"):]: torch.from_numpy(g[k]) for k in g.files if k.startswith(f"ckpt{step}_")}
        torch.save({"state_dict": {"model": sd}, "global_step": step}, os.path.join(d, f"model_ckpt_steps_{step}.ckpt"))
    loaded = {k[len("loaded_"):]: torch.from_numpy(g[k]) for k in g.files if k.startswith("loaded_")}
    mine, _ = F.load_state_dict(d, "model")
    assert sorted(mine) == sorted(loaded)
    assert all(torch.equal(mine[k], v) for k, v in loaded.items())


def test_vocoder_checkpoint_layouts(tmp_path):
    import yaml
    sd = {"conv_pre.weight_g": torch.ones(4, 1, 1), "conv_pre.weight_v": torch.randn(4, 80, 7), "conv_pre.bias": torch.zeros(4)}
    a = tmp_path / "yaml_layout"
    a.mkdir()
    yaml.safe_dump({"upsample_rates": [8, 8, 2, 2], "use_pitch_embed": True}, open(a / "config.yaml", "w"))
    torch.save({"state_dict": {"model_gen": sd, "model_disc": {}}}, a / "model_ckpt_steps_100.ckpt")
    torch.save({"state_dict": {"model_gen": {k: v * 0 for k, v in sd.items()}}}, a / "model_ckpt_steps_20.ckpt")
    got, cfg, path = F.load_vocoder_checkpoint(str(a))
    assert path.endswith("_100.ckpt") and cfg["upsample_rates"] == [8, 8, 2, 2] and torch.equal(got["conv_pre.weight_v"], sd["conv_pre.weight_v"])
    b = tmp_path / "json_layout"
    b.mkdir()
    json.dump({"upsample_rates": [8, 8, 4]}, open(b / "config.json", "w"))
    torch.save({"generator": sd}, b / "generator_v1")
    got, cfg, path = F.load_vocoder_checkpoint(str(b))
    assert path.endswith("generator_v1") and cfg["upsample_rates"] == [8, 8, 4] and sorted(got) == sorted(sd)
    with pytest.raises(FileNotFoundError):
        F.load_vocoder_checkpoint(str(tmp_path))


def _items(n=5):
    rng = np.random.default_rng(0)
    out = []
    for i in range(n):
        Fr, P = 20 + 3 * i, 4 + i
        f0 = rng.uniform(150, 400, Fr).astype(np.float32)
        f0[rng.random(Fr) < 0.3] = 0.0
        m2p = np.repeat(np.arange(1, P + 1), Fr // P + 1)[:Fr]
        out.append({"item_name": f"utt{i}", "mel": rng.normal(-3, 1, (Fr, 80)).astype(np.float32), "f0": f0, "mel2ph": m2p,
                    "ph_token": rng.integers(3, 60, P), "ep_pitches": rng.integers(48, 72, P), "ep_notedurs": rng.uniform(0.1, 0.6, P),
                    "ep_types": rng.integers(1, 3, P), "spk_embed": rng.normal(size=256).astype(np.float32),
                    "emo_embed": rng.normal(size=256).astype(np.float32)})
    return out


def test_indexed_dataset_written_by_the_reference_builder(tmp_path):
    """<prefix>.data / .idx as the reference's IndexedDatasetBuilder wrote them for _items()."""
    g = _ref()
    items = _items()
    prefix = str(tmp_path / "test")
    for ext in ("data", "idx"):
        with open(f"{prefix}.{ext}", "wb") as f:
            f.write(g["ids_" + ext].tobytes())
    with F.IndexedDatasetReader(prefix) as ds:
        assert len(ds) == len(items)
        for i in (3, 0, 4, 1, 2):
            got = ds[i]
            assert got["item_name"] == items[i]["item_name"] and np.array_equal(got["mel"], items[i]["mel"])
            assert np.array_equal(got["f0"], items[i]["f0"])
        with pytest.raises(IndexError):
            ds[len(items)]


def test_indexed_dataset_hand_written_files(tmp_path):
    items = _items(3)
    prefix = str(tmp_path / "hand")
    offs = [0]
    with open(prefix + ".data", "wb") as f:
        for it in items:
            offs.append(offs[-1] + f.write(pickle.dumps(it)))
    np.save(open(prefix + ".idx", "wb"), {"offsets": offs})
    ds = F.IndexedDatasetReader(prefix)
    assert len(ds) == 3 and np.array_equal(ds[1]["mel2ph"], items[1]["mel2ph"])
    ds.close()


def test_norm_interp_f0_matches_the_reference():
    """The reference's norm_interp_f0 (pitch_norm log, use_uv) on tracks with 0 %, some and all frames unvoiced."""
    g = _ref()
    for i in range(4):
        f0 = g[f"f0_{i}"]
        mf, mu = F.norm_interp_f0(f0.copy(), "log", True)
        assert np.array_equal(mu, g[f"f0_{i}_uv"]) and np.allclose(mf, g[f"f0_{i}_norm"], rtol=0, atol=1e-6)


def test_item_to_utterance_feeds_pack_batch():
    from stylesinger_b200.engine import pack_batch
    from stylesinger_b200.hparams import resolve
    hp = resolve(None)
    items = _items(3)
    items[1]["mel"] = np.concatenate([items[1]["mel"], np.zeros((5, 80), np.float32)])  # mel longer than mel2ph / f0
    utts = [F.item_to_utterance(it, hp) for it in items]
    u = utts[1]
    T = len(items[1]["f0"])
    assert u["ref_mels"].shape == (T, 80) and u["ref_f0"].shape == (T,) and u["mel2ph"].shape == (T,)
    assert np.isfinite(u["ref_f0"].numpy()).all() and float(u["ref_f0"].min()) > 6.0  # log2 Hz, unvoiced frames interpolated
    pb = pack_batch(utts)
    assert pb.B == 3 and int(pb.frame_offsets[-1]) == sum(len(it["f0"]) for it in items)
    assert int(pb.ph_offsets[-1]) == sum(len(it["ph_token"]) for it in items)


def test_pad_f0_to_mel_follows_the_reference_lines():
    """inference/StyleSinger.py:116-137, restated inline the way the reference writes it."""
    from stylesinger_b200.formats import pad_f0_to_mel
    rng = np.random.default_rng(0)
    for hop, pad_size in ((256, 2), (128, 4)):
        for n_mel, n_f0 in ((100, 96 - 2 * pad_size + 4), (57, 57 - 2 * pad_size), (40, 30)):
            f0 = rng.uniform(80, 800, n_f0)
            lpad = pad_size * 2
            ref = np.pad(f0, [[lpad, n_mel - len(f0) - lpad]], mode="constant")[:n_mel]
            got = pad_f0_to_mel(f0, n_mel, hop)
            assert got.shape == (n_mel,) and np.array_equal(got, ref) and (got[:lpad] == 0).all()
    with pytest.raises(AssertionError):
        pad_f0_to_mel(np.zeros(10), 20, 512)
    with pytest.raises(ValueError):      # a track longer than the mel: np.pad refuses the negative pad, as in the reference
        pad_f0_to_mel(np.zeros(30), 20, 256)


def test_preprocess_input_glue_with_stand_in_front_end():
    """StyleSingerInfer.preprocess_input: the reference's field names and call order, third-party pieces as callables.
    (The GPU pieces it calls - process_audio, emotion_embed - have their own parity tests.)"""
    from stylesinger_b200.infer import StyleSingerInfer

    class Enc:
        def encode(self, s):
            return [len(w) for w in s.split(" ")]

    eng = StyleSingerInfer.__new__(StyleSingerInfer)
    eng.hparams = {"hop_size": 256, "audio_sample_rate": 48000}
    eng.ph_encoder = Enc()
    calls = []
    eng.process_audio = lambda wav: (np.asarray(wav, np.float16), np.zeros((50, 80), np.float32))
    eng.emotion_embed = lambda w: calls.append(("emo", len(w))) or np.ones(256, np.float32)

    def pitch(wav, sr, step, fmin, fmax, thr):
        calls.append(("pitch", sr, round(step, 6), fmin, fmax, thr))
        return np.full(44, 220.0)

    inp = {"name": "x", "ph": ["a", "bb", "ccc"], "ref_audio": np.zeros(12800, np.float32)}
    out = eng.preprocess_input(inp, spk_embed_fn=lambda w: np.zeros(256, np.float32), pitch_fn=pitch,
                               preprocess_wav_fn=lambda a: a[:1000])
    assert out is inp and out["ph_token"] == [1, 2, 3] and out["item_name"] == "x" and out["mel"].shape == (50, 80)
    assert out["f0"].shape == (50,) and (out["f0"][:4] == 0).all() and (out["f0"][4:48] == 220).all() and (out["f0"][48:] == 0).all()
    assert calls == [("emo", 1000), ("pitch", 48000, round(256 / 48000, 6), 80, 800, 0.6)]
    with pytest.raises(ValueError, match="spk_embed"):
        eng.preprocess_input({"name": "y", "ph": ["a"], "ref_audio": np.zeros(10, np.float32)})
