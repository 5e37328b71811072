"""Run the UNMODIFIED reference (AaronZ345/StyleSinger) on the synthetic workload of bench.py.

Reference arms only: `bench.py --impl reference`, `tools/baseline_arms.py` (CPU figures of BASELINE.md §3 and the
GPU-PyTorch denominator of the >= 10x target) and `tests/test_gpu_reference_dropin.py`.  Nothing here is on the product
path, and nothing of this repo's engine is on the path timed here: the objects built below are the reference's own
`inference.StyleSinger.StyleSingerInfer` (its `StyleSinger` model + its registered `HifiGAN_NSF` vocoder), constructed
by the reference's own constructor from checkpoint directories written in the reference's on-disk format.

The reference source is found by tools/ref_import.py (the checkout STYLESINGER_REF names).  Inputs / checkpoints: stylesinger_b200.synth and
stylesinger_b200.hparams, which are plain Python (they do not load libstylesinger_b200.so).
"""
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)


def available():
    import ref_import
    return ref_import.find_reference() is not None


def write_checkpoints(workdir, hp):
    """exp dir, vocoder dir and processed-data dir in the layout the reference's loaders expect
    (utils/ckpt_utils.py:28-67, tasks/tts/vocoder_infer/hifigan_nsf.py:46-60, inference/StyleSinger.py:27-28)."""
    import yaml

    import ref_import
    from stylesinger_b200 import synth
    from stylesinger_b200.hparams import DEFAULT_VOCODER_CONFIG
    exp, voc, data = (os.path.join(workdir, d) for d in ("exp", "hifigan", "processed"))
    for d in (exp, voc, data):
        os.makedirs(d, exist_ok=True)
    torch.save({"state_dict": {"model": synth.acoustic_state_dict(hp, seed=0)}}, os.path.join(exp, "model_ckpt_steps_1.ckpt"))
    torch.save({"state_dict": {"model_gen": synth.vocoder_state_dict(DEFAULT_VOCODER_CONFIG, seed=0)}},
               os.path.join(voc, "model_ckpt_steps_1.ckpt"))
    with open(os.path.join(voc, "config.yaml"), "w") as f:
        yaml.safe_dump(dict(DEFAULT_VOCODER_CONFIG), f)
    shutil.copyfile(os.path.join(ref_import.find_reference(), "ZH_checkpoint_phone_set.json"), os.path.join(data, "phone_set.json"))
    return exp, voc, data


class ReferenceRunner:
    """The reference's StyleSingerInfer on `device` ('cpu' or 'cuda') with synthetic checkpoints."""

    def __init__(self, T=100, device="cpu", threads=None):
        import ref_import
        if threads:
            torch.set_num_threads(int(threads))
        self.workdir = tempfile.mkdtemp(prefix="ssb_ref_")
        from stylesinger_b200.hparams import resolve
        exp, voc, data = write_checkpoints(self.workdir, resolve(timesteps=T, K_step=T, f0_timesteps=T))
        self.hp = ref_import.install(T=T, overrides={"exp_name": exp, "vocoder_ckpt": voc, "processed_data_dir": data,
                                                      "work_dir": exp})
        import modules.diff.gaussian_multinomial_diffusion as gmd
        import modules.diff.shallow_diffusion_tts as sdt
        sdt.tqdm = lambda it, **k: it  # progress bars off; no arithmetic touched
        gmd.tqdm = lambda it, **k: it
        import inference.StyleSinger as I
        self.device = device
        self.I = I
        real = torch.cuda.is_available
        if device == "cpu":
            # tasks/tts/vocoder_infer/hifigan_nsf.py:27 picks cuda whenever it is visible: hide it while the CPU arm's
            # vocoder wrapper is constructed (it keeps the device it chose then)
            torch.cuda.is_available = lambda: False
        try:
            self.infer = I.StyleSingerInfer(self.hp, device=device)
        finally:
            torch.cuda.is_available = real

    def close(self):
        shutil.rmtree(self.workdir, ignore_errors=True)

    @staticmethod
    def item_from_utterance(u):
        """synth.make_utterance dict -> the item dict `preprocess_input` produces (inference/StyleSinger.py:94-137).
        `f0` is raw Hz there (norm_interp_f0 is applied by input_to_batch, :152); the synthetic ref_f0 is log2 Hz with no
        unvoiced frame, so 2**ref_f0 is the Hz track that maps back onto it."""
        return {"item_name": "synth", "ph": "", "ph_token": u["txt_tokens"].numpy(), "note": u["note"].numpy(),
                "note_dur": u["note_dur"].numpy(), "note_type": u["note_type"].numpy(),
                "spk_embed": u["spk_embed"].numpy(), "emo_embed": u["emo_embed"].numpy(),
                "mel": u["ref_mels"].numpy(), "f0": np.exp2(u["ref_f0"].numpy().astype(np.float64)).astype(np.float32)}

    def forward_model(self, item, mel2ph=None):
        """mel2ph None: the stock `StyleSingerInfer.forward_model` (predicted durations).  With mel2ph: the same lines
        (inference/StyleSinger.py:41-64) with `mel2ph=` handed to `StyleSinger.forward`, so that the frame count equals
        the bench workload's (the b200 arm feeds the same explicit mel2ph).  Returns the waveform (np.float32)."""
        inf, hp = self.infer, self.hp
        with torch.no_grad():
            if mel2ph is None:
                return inf.forward_model(item)
            s = inf.input_to_batch(item)
            out = inf.model(s["txt_tokens"], mel2ph=torch.as_tensor(mel2ph).long()[None].to(inf.device), spk_embed=s["spk_embed"],
                            emo_embed=s["emo_embed"], ref_mels=s["mels"], ref_f0=s["f0"], global_steps=320000, infer=True,
                            note=s["notes"], note_dur=s["note_durs"], note_type=s["note_types"])
            f0 = out["f0_denorm"].cpu().numpy()
            mel = out["mel_out"].cpu().detach().numpy()
            mask = np.abs(mel).sum(-1) > 0
            mel = np.clip(mel[mask], hp["mel_vmin"], hp["mel_vmax"])
            f0 = f0[:len(mask)] if len(f0) > len(mask) else f0
            return inf.vocoder.spec2wav(mel, f0=f0[mask])

    def timed_pass(self, seconds, utt_idx=0, explicit_mel2ph=True):
        """One ph -> mel -> wav pass over one synthetic utterance: (frames, elapsed seconds)."""
        from stylesinger_b200 import synth
        u = synth.make_utterance(seconds, utt_idx=utt_idx)
        item = self.item_from_utterance(u)
        if self.device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        wav = self.forward_model(item, u["mel2ph"].numpy() if explicit_mel2ph else None)
        if self.device != "cpu":
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return int(len(wav) // 256), dt


if __name__ == "__main__":  # quick self-check: python baseline/ref_harness.py [seconds] [T] [device]
    secs = float(sys.argv[1]) if len(sys.argv) > 1 else 0.5
    T = int(sys.argv[2]) if len(sys.argv) > 2 else 4
    dev = sys.argv[3] if len(sys.argv) > 3 else "cpu"
    r = ReferenceRunner(T=T, device=dev, threads=8)
    print(json.dumps({"frames_dt": r.timed_pass(secs), "stock_forward_model_frames_dt": r.timed_pass(secs, explicit_mel2ph=False)}))
    r.close()
