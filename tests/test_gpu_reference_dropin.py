"""This repo's drop-ins for the reference's extension points (SURVEY.md section 8b) against what the unmodified reference
computed at those points.  tests/golden/ref_dropin_T8.npz (tools/make_golden.py dropin) holds one run of the reference's
own `inference.StyleSinger.StyleSingerInfer.forward_model` (T=8, predicted durations, use_nsf off, torch.randn* patched to
one seeded NoiseSource stream): the inputs and outputs of its model call, the first and last call of every module a
registry-level drop-in replaces (both DDiffNets, DIFF_DECODERS['wavenet'], FS_ENCODERS / FS_DECODERS 'fft', get_style),
and the vocoder's input and waveform.  Arrays that were identical in that run are stored once (meta["alias"]).
The tests call the drop-ins on those recorded inputs and compare with the recorded outputs; the reference's own code
(its registries, sampler loops and inference driver) is not run here.
"""
import numpy as np
import pytest
import torch
import yaml

from tests.common import golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def ref():
    g, meta = golden("ref_dropin_T8")
    a = {k: g[k] for k in g.files if k != "meta"}
    a.update({k: a[v] for k, v in meta["alias"].items()})
    return a, meta


@pytest.fixture(scope="module")
def engine(ref):
    from stylesinger_b200 import synth
    from stylesinger_b200.engine import AcousticModel
    from stylesinger_b200.hparams import resolve
    T = ref[1]["T"]
    hp = resolve(timesteps=T, K_step=T, f0_timesteps=T)
    return AcousticModel(synth.acoustic_state_dict(hp, seed=0), hp, DEV)  # the checkpoint the reference run loaded


def _maxabs(a, b):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max())


def _vocoder(tmp_path, use_nsf):
    """The HiFi-GAN drop-in built from a checkpoint directory in the reference's on-disk layout (config.yaml +
    model_ckpt_steps_*.ckpt with a 'model_gen' state dict), as the reference's vocoder loader reads it."""
    from stylesinger_b200 import formats, synth
    from stylesinger_b200.hparams import DEFAULT_VOCODER_CONFIG
    from stylesinger_b200.modules import HifiGAN
    d = tmp_path / "hifigan"
    d.mkdir()
    torch.save({"state_dict": {"model_gen": synth.vocoder_state_dict(DEFAULT_VOCODER_CONFIG, seed=0)}}, d / "model_ckpt_steps_1.ckpt")
    with open(d / "config.yaml", "w") as f:
        yaml.safe_dump(dict(DEFAULT_VOCODER_CONFIG), f)
    sd, cfg, _ = formats.load_vocoder_checkpoint(str(d))
    return HifiGAN(sd, cfg, DEV, use_nsf=use_nsf)


def test_registry_level_dropins_match_the_reference_modules(ref, engine):
    """Each registry-level drop-in called on the inputs the reference's own module received inside forward_model (first
    and last reverse step for the three denoisers) must return what that module returned."""
    from stylesinger_b200 import modules as M
    a, meta = ref

    def t(k):
        return torch.from_numpy(a[k]).to(DEV)

    facade = M.StyleSinger(engine=engine, hparams=engine.hp)
    err = {}
    with torch.no_grad():
        err["encoder"] = _maxabs(M.FastspeechEncoder(engine)(t("encoder0_a0")), a["encoder0_out"])
        err["decoder"] = _maxabs(M.FastspeechDecoder(engine)(t("decoder0_a0")), a["decoder0_out"])
        style = facade.get_style(t("get_style0_a0"), t("get_style0_a1"), {"ref_f0": t("get_style0_a2")}, True, meta["global_steps"])
        err["get_style"] = _maxabs(style, a["get_style0_out"])
        for i in (0, 1):
            err[f"diffnet{i}"] = _maxabs(M.DiffNet(engine)(t(f"diffnet{i}_a0"), t(f"diffnet{i}_a1"), cond=t(f"diffnet{i}_k_cond")),
                                         a[f"diffnet{i}_out"])
            for which in (1, 2):
                k = f"ddiffnet{which}{i}"
                err[k] = _maxabs(M.DDiffNet(engine, which)(*(t(f"{k}_a{j}") for j in range(5))), a[f"{k}_out"])
    print("drop-ins vs reference modules (L-inf):", {k: f"{v:.3e}" for k, v in err.items()})
    assert all(v < 1e-3 for v in err.values()), err


def test_whole_model_dropin_on_the_reference_model_call(ref, engine, tmp_path):
    """INTEGRATION.md section 2.1: modules.StyleSinger called the way the reference's StyleSingerInfer.forward_model calls
    self.model (its input_to_batch tensors, predicted durations, global_steps, infer=True) on the draws the reference
    consumed.  The reference does not drive it here: forward_model's post-processing (inference/StyleSinger.py:52-63:
    drop all-zero frames, clip to [mel_vmin, mel_vmax]) is restated below, and the vocoder drop-in makes the waveform."""
    from stylesinger_b200 import modules as M
    from tests.common import engine_noise_from_stream
    a, meta = ref
    T, seed = meta["T"], meta["seed"]

    class Injected(M.StyleSinger):  # same draws as the reference run: SURVEY A.10 order, sized by the predicted frame count
        def forward(self, *args, **k):
            k["noise"] = lambda fo: engine_noise_from_stream(seed, T, T, int(fo[-1]), DEV)[0]
            return super().forward(*args, **k)

    def t(k):
        return torch.from_numpy(a["in_" + k]).to(DEV)

    model = Injected(engine=engine, hparams=engine.hp)
    with torch.no_grad():
        ret = model(t("txt_tokens"), spk_embed=t("spk_embed"), emo_embed=t("emo_embed"), ref_mels=t("ref_mels"), ref_f0=t("ref_f0"),
                    global_steps=meta["global_steps"], infer=True, note=t("note"), note_dur=t("note_dur"), note_type=t("note_type"))
    assert np.array_equal(ret["mel2ph"].cpu().numpy(), a["ret_mel2ph"])
    f0_pred = ret["f0_denorm"].cpu().numpy()
    mel_pred = ret["mel_out"].cpu().numpy()
    mask = np.abs(mel_pred).sum(-1) > 0
    mel_pred = np.clip(mel_pred[mask], meta["mel_vmin"], meta["mel_vmax"])
    wav = _vocoder(tmp_path, use_nsf=False).spec2wav(mel_pred, f0=f0_pred[:len(mask)][mask])
    e_mel = _maxabs(ret["mel_out"], a["ret_mel_out"])
    e_wav = _maxabs(wav, a["wav"])
    print(f"whole-model drop-in on the reference model call: mel L-inf {e_mel:.3e}, wav {e_wav:.3e}")
    assert e_mel < 1e-3 and e_wav < 2e-3
    for k in ("style", "decoder_inp", "pitch_pred"):
        assert _maxabs(ret[k], a["ret_" + k]) < 1e-3, k


def test_vocoder_registry_dropin(ref, tmp_path):
    """INTEGRATION.md section 2.3: modules.HifiGAN, the vocoder meant for the reference's 'HifiGAN_NSF' registry slot,
    built from a checkpoint directory in the reference's layout, turns the mel the reference's forward_model handed to
    its vocoder into the reference's waveform.  f0 is not passed: with use_nsf off the reference's vocoder ignores it.
    Registering the class in the reference's registry is not exercised."""
    a, _ = ref
    wav = _vocoder(tmp_path, use_nsf=False).spec2wav(a["vocoder0_a0"], f0=None)
    e = _maxabs(wav, a["wav"])
    print(f"reference mel + B200 vocoder drop-in: wav L-inf {e:.3e}")
    assert e < 1e-3
