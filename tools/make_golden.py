"""Generate tests/golden/*.npz by executing the UNMODIFIED reference.

    STYLESINGER_REF=<checkout of AaronZ345/StyleSinger> python tools/make_golden.py [case ...]   # writes tests/golden/

What it does (SURVEY.md §8c): imports the reference through tools/ref_import.py, builds the
reference's own ``StyleSinger`` / ``HifiGanGenerator`` modules, loads the synthetic checkpoints of
``stylesinger_b200.synth`` with ``strict=True`` (which also proves state-dict name/shape
compatibility with released checkpoints), monkey-patches ``torch.randn/randn_like/rand/rand_like``
to a seeded ``NoiseSource`` so the stochastic samplers are reproducible, runs the reference and
dumps small fixtures.  The fixtures pin oracle/stylesinger_oracle.py (tests/test_oracle_golden.py)
and, through it and directly, the CUDA path (tests/test_gpu_*.py).
"""
import contextlib
import json
import os
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))

from oracle.stylesinger_oracle import NoiseSource  # noqa: E402
from stylesinger_b200 import synth  # noqa: E402
from stylesinger_b200.hparams import DEFAULT_VOCODER_CONFIG  # noqa: E402

OUT = os.path.join(REPO, "tests", "golden")


@contextlib.contextmanager
def patched_rng(ns):
    o = (torch.randn, torch.randn_like, torch.rand, torch.rand_like)

    def _shape(a):
        if len(a) == 1 and isinstance(a[0], (tuple, list, torch.Size)):
            return tuple(a[0])
        return tuple(a)

    torch.randn = lambda *a, **k: ns.randn(_shape(a))
    torch.randn_like = lambda x, **k: ns.randn(tuple(x.shape))
    torch.rand = lambda *a, **k: ns.rand(_shape(a))
    torch.rand_like = lambda x, **k: ns.rand(tuple(x.shape))
    try:
        yield
    finally:
        torch.randn, torch.randn_like, torch.rand, torch.rand_like = o


class _Dict:
    def pad(self):
        return 0

    def __len__(self):
        return synth.N_TOKENS


def build_reference_model(T, f0_T=None):
    import ref_import
    hp = ref_import.install(T=T, f0_T=f0_T)
    # fresh import state for every T: the schedule buffers are built in __init__
    import modules.diff.shallow_diffusion_tts as sdt
    import modules.diff.gaussian_multinomial_diffusion as gmd
    sdt.tqdm = lambda it, **k: it
    gmd.tqdm = lambda it, **k: it
    from modules.StyleSinger.stylesinger import StyleSinger
    model = StyleSinger(_Dict()).eval()
    sd = synth.acoustic_state_dict(dict(hp), seed=0)
    missing, unexpected = model.load_state_dict(sd, strict=True), None
    return model, hp, sd


def batchify(u):
    return dict(txt_tokens=u["txt_tokens"][None], note=u["note"][None], note_dur=u["note_dur"][None],
                note_type=u["note_type"][None], spk_embed=u["spk_embed"][None], emo_embed=u["emo_embed"][None],
                ref_mels=u["ref_mels"][None], ref_f0=u["ref_f0"])  # ref_f0 is 1-D at B=1 (inference/StyleSinger.py:151)


def run_model(model, u, seed, mel2ph=True, global_steps=320000):
    ns = NoiseSource(seed)
    b = batchify(u)
    cap = {}
    h = model.style_extractor.rqvae.register_forward_hook(lambda m, i, o: cap.__setitem__("rq_in", i[0].detach().clone()))
    with torch.no_grad(), patched_rng(ns):
        out = model(b["txt_tokens"], mel2ph=u["mel2ph"][None] if mel2ph else None, spk_embed=b["spk_embed"],
                    emo_embed=b["emo_embed"], ref_mels=b["ref_mels"].clone(), ref_f0=b["ref_f0"].clone(),
                    global_steps=global_steps, infer=True, note=b["note"], note_dur=b["note_dur"],
                    note_type=b["note_type"])
        codes = model.style_extractor.rqvae.quantize(cap["rq_in"])[1]
    h.remove()
    out["rq_codes"] = codes
    out["rq_in"] = cap["rq_in"]
    return out, ns.log


def np32(t):
    return t.detach().cpu().numpy().astype(np.float32)


def case_model(name, T, frames, phones, ref_frames, seed, utt_idx, with_dur_case=True):
    model, hp, sd = build_reference_model(T)
    u = synth.make_utterance(frames / 187.5, utt_idx=utt_idx, ref_frames=ref_frames, frames=frames, phones=phones)
    out, log = run_model(model, u, seed)
    coarse, _ = run_model(model, u, seed, global_steps=50000)  # forcing < global_steps < diff_start: coarse mel only
    d = {
        "meta": json.dumps({"T": T, "frames": frames, "phones": phones, "ref_frames": ref_frames, "seed": seed,
                            "utt_idx": utt_idx, "noise_log": log}),
        "style": np32(out["style"][0]), "rq_codes": out["rq_codes"][0].numpy().astype(np.int64),
        "rq_in": np32(out["rq_in"][0]),
        "pitch_pred": np32(out["pitch_pred"][0]), "f0_denorm": np32(out["f0_denorm"][0]),
        "decoder_inp": np32(out["decoder_inp"][0]), "coarse_mel": np32(coarse["mel_out"][0]),
        "mel_out": np32(out["mel_out"][0]), "spk_embed": np32(out["spk_embed"][0]), "emo_embed": np32(out["emo_embed"][0]),
    }
    if with_dur_case:
        o2, log2 = run_model(model, u, seed + 1, mel2ph=False)
        d.update({"dur_mel2ph": o2["mel2ph"][0].numpy().astype(np.int64), "dur_logdur": np32(o2["dur"][0]),
                  "dur_mel_out": np32(o2["mel_out"][0]), "dur_f0_denorm": np32(o2["f0_denorm"][0]),
                  "dur_noise_log": json.dumps(log2)})
    # single denoiser evaluations (deterministic)
    g = torch.Generator().manual_seed(99)
    Fr = 48
    spec = torch.randn(1, 1, 80, Fr, generator=g)
    cond = torch.randn(1, 256, Fr, generator=g)
    with torch.no_grad():
        e1 = model.postdiff.denoise_fn(spec, torch.tensor([T - 1]), cond)
        f0 = torch.randn(1, 1, Fr, generator=g)
        uv = (torch.rand(1, Fr, generator=g) < 0.4).long()
        e2 = model.gm_diffnet(f0, uv, torch.tensor([1]), cond, torch.ones(1, Fr))
        e3 = model.gm_diffnet_inpainte(f0, uv, torch.tensor([0]), cond, torch.ones(1, Fr))
    d.update({"dn_spec": np32(spec[0, 0]), "dn_cond": np32(cond[0]), "dn_out": np32(e1[0, 0]),
              "dd_f0": np32(f0[0, 0]), "dd_uv": uv[0].numpy().astype(np.int64), "dd_out": np32(e2[0]),
              "dd_out_inp": np32(e3[0])})
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
    print("wrote", name, {k: (v.shape if hasattr(v, "shape") else "meta") for k, v in d.items()})


def case_vocoder(name, frames, seed):
    import ref_import
    ref_import.install(T=4)
    from modules.hifigan.hifigan_nsf import HifiGanGenerator
    h = dict(DEFAULT_VOCODER_CONFIG)
    vsd = synth.vocoder_state_dict(h, seed=0)
    gen = HifiGanGenerator(h)
    gen.load_state_dict(vsd, strict=True)
    gen.remove_weight_norm()
    gen.eval()
    g = torch.Generator().manual_seed(seed)
    mel = (-3.0 + 0.8 * torch.randn(frames, 80, generator=g)).clamp(-6, 1.5)
    f0 = 150 + 350 * torch.rand(frames, generator=g)
    f0[frames // 3: frames // 3 + 5] = 0  # an unvoiced stretch
    ns = NoiseSource(seed + 5)
    with torch.no_grad(), patched_rng(ns):
        c = torch.FloatTensor(mel.numpy()).unsqueeze(0).transpose(2, 1)
        y = gen(c, torch.FloatTensor(f0.numpy()[None, :])).view(-1)
        ns2 = NoiseSource(seed + 6)
    with torch.no_grad():
        y_nof0 = gen(c).view(-1)
    d = {"meta": json.dumps({"frames": frames, "seed": seed, "noise_log": ns.log}), "mel": np32(mel), "f0": np32(f0),
         "wav": np32(y), "wav_nof0": np32(y_nof0)}
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
    print("wrote", name, y.shape, float(y.abs().max()), float(y.std()))


def case_plms(name, T=100, interval=10, frames=48, seed=61):
    """f2: the reference's PLMS sampler (GaussianDiffusion.p_sample_plms, shallow_diffusion_tts.py:164-197) driven exactly
    as GaussianDiffusion.forward does under hparams['pndm_speedup'] (:254-260), on the StyleSinger mel denoiser (the
    DiffusionDecoder instance inherits the method)."""
    from collections import deque
    model, hp, sd = build_reference_model(T)
    pd = model.postdiff
    g = torch.Generator().manual_seed(seed)
    cond = torch.randn(1, frames, 256, generator=g)
    coarse = (-3 + 0.8 * torch.randn(1, frames, 80, generator=g)).clamp(-6, 0.5)
    ns = NoiseSource(seed + 1)
    with torch.no_grad(), patched_rng(ns):
        c = cond.transpose(1, 2)
        fs2 = pd.norm_spec(coarse).transpose(1, 2)[:, None, :, :]
        x = pd.q_sample(x_start=fs2, t=torch.tensor([T - 1]).long())
        pd.noise_list = deque(maxlen=4)
        for i in reversed(range(0, T, interval)):
            x = pd.p_sample_plms(x, torch.full((1,), i, dtype=torch.long), interval, c)
        mel = pd.denorm_spec(x[:, 0].transpose(1, 2))
    d = {"meta": json.dumps({"T": T, "interval": interval, "frames": frames, "seed": seed, "noise_log": ns.log}),
         "cond": np32(cond[0]), "coarse": np32(coarse[0]), "mel": np32(mel[0])}
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
    print("wrote", name, mel.shape, float(mel.abs().max()))


def case_schedules(name, Ts=(4, 25, 50, 100, 200, 500)):
    """Registered schedule buffers of the reference's DiffusionDecoder / GaussianMultinomialDiffusion at several T
    (shallow_diffusion_tts.py:86-119, gaussian_multinomial_diffusion.py:237-283): pins the oracle's and the product's
    independently written schedule code, incl. the T values of BASELINE.json configs[4]."""
    gk = ["betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod",
          "log_one_minus_alphas_cumprod", "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_variance",
          "posterior_log_variance_clipped", "posterior_mean_coef1", "posterior_mean_coef2"]
    mk = ["log_alpha", "log_1_min_alpha", "log_cumprod_alpha", "log_1_min_cumprod_alpha"]
    d = {"Ts": np.asarray(Ts, np.int64)}
    for T in Ts:
        model, hp, _ = build_reference_model(T)
        for k in gk:
            d[f"mel_T{T}_{k}"] = np32(getattr(model.postdiff, k))
            d[f"f0_T{T}_{k}"] = np32(getattr(model.f0_gen, k))
        for k in mk:
            d[f"f0_T{T}_{k}"] = np32(getattr(model.f0_gen, k))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
    print("wrote", name, len(d), "arrays")


def case_emotion_encoder(name, partials=5, seed=71):
    """f3: the reference's own EmotionEncoder (data_gen/tts/emotion/model.py:10-77, the network behind `emo_embed`,
    inference/StyleSinger.py:106) with seeded random weights on seeded random 160-frame x 40-channel partials:
    `inference` (= hidden[-1], what data_gen/tts/emotion/inference.py:54 uses), `forward` (relu(linear) L2-normalised) and
    the utterance embedding of embed_utterance (inference.py:150-151: mean of the partial embeddings, L2-normalised)."""
    import ref_import
    ref_import.install(T=4)  # reference on sys.path + import shims (hparams unused by the encoder)
    from data_gen.tts.emotion.model import EmotionEncoder
    from oracle.frontend_oracle import emotion_encoder_weights
    cpu = torch.device("cpu")
    model = EmotionEncoder(cpu, cpu).eval()
    # weights: numpy legacy RandomState stream (stable across versions), loaded the stock way; the fixture then only holds
    # inputs and outputs and the tests regenerate the same weights from the seed
    sd = emotion_encoder_weights(seed)
    missing = model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=False)
    assert not [k for k in missing.missing_keys if k.startswith(("lstm.", "linear."))], missing
    g = torch.Generator().manual_seed(seed + 1)
    frames = (torch.randn(partials, 160, 40, generator=g).abs() * 0.3).float()
    with torch.no_grad():
        hidden = model.inference(frames)
        embeds = model.forward(frames)
        frames2 = (torch.randn(3, 97, 40, generator=g).abs() * 2.0).float()  # another length, louder input
        hidden2 = model.inference(frames2)
    raw = hidden.numpy().mean(axis=0)
    d = {"frames2": np32(frames2), "hidden2": np32(hidden2), "seed": np.int64(seed), "frames": np32(frames), "hidden": np32(hidden), "embeds": np32(embeds),
         "utt_embed": (raw / np.linalg.norm(raw, 2)).astype(np.float32)}
    # partial-utterance slicing (inference.py:58-107) for a spread of lengths incl. the short / coverage-edge cases
    from data_gen.tts.emotion.inference import compute_partial_slices
    ns = [1, 159, 160, 8000, 19199, 19200, 25599, 25600, 31999, 32000, 38400, 44799, 44800, 48000, 160000, 163840, 479999]
    rows = []
    for n in ns:
        wav_sl, mel_sl = compute_partial_slices(n)
        for w, m in zip(wav_sl, mel_sl):
            rows.append([n, w.start, w.stop, m.start, m.stop])
    d["slices"] = np.asarray(rows, np.int64)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
    print("wrote", name, len(d), "arrays")


def _put(d, alias, key, t):
    """Store t under key, or record key as an alias of an identical array already stored (keeps the fixture small)."""
    a = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
    for k, v in d.items():
        if isinstance(v, np.ndarray) and v.dtype == a.dtype and v.shape == a.shape and np.array_equal(v, a):
            alias[key] = k
            return
    d[key] = a


def case_dropin(name, T=8, seed=2024, utt=dict(seconds=0.3, utt_idx=11, ref_frames=32, phones=4)):
    """The reference's own StyleSingerInfer.forward_model (predicted durations, use_nsf off, torch.randn* on
    NoiseSource(seed)) on one synthetic item, recorded where stylesinger_b200.modules plugs in: the model call's inputs and
    outputs, the first and last call of every module a registry-level drop-in replaces, and the vocoder's input and
    waveform (tests/test_gpu_reference_dropin.py)."""
    sys.path.insert(0, os.path.join(REPO, "baseline"))
    import ref_harness
    r = ref_harness.ReferenceRunner(T=T, device="cpu")
    r.hp["use_nsf"] = False
    u = synth.make_utterance(utt["seconds"], utt_idx=utt["utt_idx"], ref_frames=utt["ref_frames"], phones=utt["phones"])
    item = r.item_from_utterance(u)
    m = r.infer.model
    calls = {}
    hooks = []
    for key, mod in (("model", m), ("encoder", m.encoder), ("decoder", m.decoder), ("diffnet", m.postdiff.denoise_fn),
                     ("ddiffnet1", m.f0_gen._denoise_fn), ("ddiffnet2", m.f0_gen_inpainte._denoise_fn)):
        hooks.append(mod.register_forward_hook(lambda mod_, a, k, o, key=key: calls.setdefault(key, []).append((a, k, o)),
                                               with_kwargs=True))
    get_style, spec2wav = m.get_style, r.infer.vocoder.spec2wav

    def style_spy(encoder_out, ref_mels, ret, infer=False, global_steps=0):
        out = get_style(encoder_out, ref_mels, ret, infer, global_steps)
        calls.setdefault("get_style", []).append(((encoder_out.clone(), ref_mels.clone(), ret["ref_f0"].clone()), {}, out))
        return out

    def voc_spy(mel, **kw):
        wav = spec2wav(mel, **kw)
        calls["vocoder"] = [((torch.from_numpy(mel.copy()),), {}, torch.from_numpy(np.asarray(wav)))]
        return wav

    m.get_style, r.infer.vocoder.spec2wav = style_spy, voc_spy
    with torch.no_grad(), patched_rng(NoiseSource(seed)):
        wav = r.infer.forward_model(item)
    for h in hooks:
        h.remove()
    r.close()
    (ma, mk, ret), = calls.pop("model")
    mk = dict(mk, txt_tokens=ma[0])
    d, alias = {"wav": np.asarray(wav, np.float32)}, {}
    for k in ("txt_tokens", "spk_embed", "emo_embed", "ref_mels", "ref_f0", "note", "note_dur", "note_type"):
        _put(d, alias, "in_" + k, mk[k])
    for k in ("mel2ph", "mel_out", "f0_denorm", "style", "decoder_inp", "pitch_pred"):
        _put(d, alias, "ret_" + k, ret[k])
    for key, cs in calls.items():
        for i, (a, kw, o) in ((0, cs[0]), (1, cs[-1])) if len(cs) > 1 else ((0, cs[0]),):
            for j, t in enumerate(a):
                _put(d, alias, f"{key}{i}_a{j}", t)
            for k, t in kw.items():
                _put(d, alias, f"{key}{i}_k_{k}", t)
            _put(d, alias, f"{key}{i}_out", o)
    d["meta"] = json.dumps({"T": T, "seed": seed, "utt": utt, "global_steps": mk["global_steps"], "mel_vmin": r.hp["mel_vmin"],
                            "mel_vmax": r.hp["mel_vmax"], "calls": {k: len(v) for k, v in calls.items()}, "alias": alias})
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
    print("wrote", name, {k: v.shape for k, v in d.items() if hasattr(v, "shape")}, json.loads(d["meta"]))


def case_formats(name):
    """The reference's own on-disk writers and pure host helpers on small seeded inputs (tests/test_formats_cpu.py):
    utils/commons/indexed_datasets.py's builder output, utils/commons/ckpt_utils.py's load_ckpt choice among two
    checkpoints, and utils/pitch_utils.py's norm_interp_f0."""
    import importlib.util
    import pickle
    import tempfile
    import types
    import ref_import
    sys.path.insert(0, os.path.join(REPO, "tests"))

    def ref_module(rel, stubs=()):
        for s in stubs:
            sys.modules.setdefault(s, types.ModuleType(s))
        spec = importlib.util.spec_from_file_location("ref_" + os.path.basename(rel)[:-3], os.path.join(ref_import.REF, rel))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    from test_formats_cpu import _items
    d = {}
    tmp = tempfile.mkdtemp(prefix="ssb_golden_")
    ids = ref_module("utils/commons/indexed_datasets.py")
    b = ids.IndexedDatasetBuilder(os.path.join(tmp, "test"))
    for it in _items():
        b.add_item(it)
    b.finalize()
    for ext in ("data", "idx"):
        d["ids_" + ext] = np.frombuffer(open(os.path.join(tmp, "test." + ext), "rb").read(), np.uint8)

    ck = ref_module("utils/commons/ckpt_utils.py")

    class Tiny(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.encoder = torch.nn.Linear(4, 3)
            self.proj = torch.nn.Conv1d(3, 2, 3)

    torch.manual_seed(0)
    for step in (7, 3):
        sd = Tiny().state_dict()
        torch.save({"state_dict": {"model": sd}, "global_step": step}, os.path.join(tmp, f"model_ckpt_steps_{step}.ckpt"))
        d.update({f"ckpt{step}_{k}": v.numpy() for k, v in sd.items()})
    dst = Tiny()
    ck.load_ckpt(dst, tmp, "model", strict=True)
    d.update({f"loaded_{k}": v.numpy() for k, v in dst.state_dict().items()})

    pu = ref_module("utils/pitch_utils.py", stubs=("librosa",))
    rng = np.random.default_rng(1)
    hp = {"pitch_norm": "log", "use_uv": True}
    for i, (n, p0) in enumerate(((50, 0.3), (17, 0.0), (9, 1.0), (64, 0.9))):
        f0 = rng.uniform(100, 600, n).astype(np.float32)
        f0[rng.random(n) < p0] = 0.0
        rf, ru = pu.norm_interp_f0(f0.copy(), hp)
        d.update({f"f0_{i}": f0, f"f0_{i}_norm": rf.numpy(), f"f0_{i}_uv": ru.numpy()})
    import shutil
    shutil.rmtree(tmp)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)
    print("wrote", name, len(d), "arrays")


if __name__ == "__main__":
    sys.dont_write_bytecode = True  # importing the reference must not write __pycache__ into its tree
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    which = sys.argv[1:] or ["small", "t25", "t100", "plms", "sched", "voc", "emo", "dropin", "formats"]
    if "small" in which:
        case_model("ref_small_T4", T=4, frames=96, phones=12, ref_frames=64, seed=11, utt_idx=100)
    if "t25" in which:
        case_model("ref_f64_T25", T=25, frames=64, phones=8, ref_frames=48, seed=21, utt_idx=101, with_dur_case=False)
    if "t100" in which:  # the bench's step count (T=100 mel + 2 x 100 F0 steps) on a tiny utterance
        case_model("ref_f32_T100", T=100, frames=32, phones=4, ref_frames=32, seed=41, utt_idx=102, with_dur_case=False)
    if "plms" in which:
        case_plms("ref_plms_T100_i10")
    if "sched" in which:
        case_schedules("ref_schedules")
    if "voc" in which:
        case_vocoder("ref_vocoder_f24", frames=24, seed=31)
    if "emo" in which:
        case_emotion_encoder("ref_emotion_encoder")
    if "dropin" in which:
        case_dropin("ref_dropin_T8")
    if "formats" in which:
        case_formats("ref_formats")
