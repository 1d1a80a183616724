"""ORACLE PINNING against vectors produced by EXECUTING the reference's own source files (tests/golden/reference_exec.npz,
generated in the build container by tests/golden/make_reference_vectors.py — see its header for what is executed as-is and what
is substituted). CPU tests: the oracle reproduces them. GPU tests: the CUDA path reproduces them with no oracle in the loop.

Bars: integer / index results bit-exact; float64 numpy paths exact to 1e-12; float32 tensor paths to a few ulp (1e-6 relative);
losses to 1e-5 relative (float32 reduction order)."""
import json
import os

import numpy as np
import pytest
import torch

from hparams import hparams

HERE = os.path.dirname(os.path.abspath(__file__))
R = np.load(os.path.join(HERE, "golden", "reference_exec.npz"))


# ------------------------------------------------------------------------------------------------ hparams
def test_hparams_defaults_equal_the_reference_values():
    """every scalar / list default of the reference's hparams.py (captured when its module was imported) is present here with
    the same value"""
    ref = json.load(open(os.path.join(HERE, "golden", "reference_hparams.json")))
    ours = hparams.values()
    missing = [k for k in ref if k not in ours]
    assert not missing, missing
    diff = {k: (ref[k], ours[k]) for k in ref if (list(ours[k]) if isinstance(ours[k], (list, tuple)) else ours[k]) != ref[k]}
    assert not diff, diff
    assert len(ref) > 150


# ------------------------------------------------------------------------------------------------ mu-law family
def test_oracle_mulaw_float64_matches_reference_numpy_path():
    from oracle import audio as oa
    x = R["mulaw_x64"]
    assert np.array_equal(oa.mulaw_quantize(x).astype(np.int32), R["mulaw_q_f64"])          # incl. both sides of all 254 bin edges
    assert np.abs(oa.mulaw(x) - R["mulaw_f64"]).max() < 1e-15
    assert np.abs(oa.inv_mulaw(R["mulaw_f64"]) - R["inv_mulaw_f64"]).max() < 1e-15
    assert R["mulaw_q_scalar0"].tolist() == [127, 127] == [int(oa.mulaw_quantize(np.float64(0))), int(oa.mulaw_quantize(np.float32(0)))]


def test_oracle_mulaw_float32_matches_reference_tensor_path():
    """the production dtype (librosa.load gives float32; numpy 1.14 kept float32 throughout, as the reference's tensor path does)"""
    from oracle import audio as oa
    x = R["mulaw_x32"]
    q = oa.mulaw_quantize(x).astype(np.int32)
    assert np.array_equal(q, R["mulaw_q_tensor_f32"])
    assert np.abs(oa.mulaw(x) - R["mulaw_tensor_f32"]).max() <= 2 ** -23            # <= 1 ulp at 1.0: torch log1pf vs the correctly rounded definition
    assert np.abs(oa.inv_mulaw(R["mulaw_tensor_f32"]) - R["inv_mulaw_tensor_f32"]).max() <= 2e-7
    assert np.abs(oa.inv_mulaw_quantize(np.arange(256)) - R["inv_mulaw_q_tensor_all"]).max() <= 2e-7
    assert np.abs(oa.inv_mulaw_quantize(np.arange(256)) - R["inv_mulaw_q_all"]).max() <= 2e-7
    # for the record: numpy >= 2 promotes the reference's numpy float32 path to float64 at `/ np.log1p(255)`; that changes a
    # handful of indices that sit within one float32 ulp of a bin edge and nothing else
    d = R["mulaw_q_numpy_f32_numpy2"] != R["mulaw_q_tensor_f32"]
    assert d[-2000:].mean() < 1e-4 and np.abs(R["mulaw_q_numpy_f32_numpy2"][d] - R["mulaw_q_tensor_f32"][d]).max(initial=0) <= 1


@pytest.mark.gpu
def test_cuda_mulaw_matches_reference_tensor_path():
    from t2_import import t2
    x = torch.from_numpy(R["mulaw_x32"]).cuda()
    assert np.array_equal(t2.audio.mulaw_quantize(x).cpu().numpy(), R["mulaw_q_tensor_f32"])         # bit-exact indices
    assert np.abs(t2.audio.mulaw(x).cpu().numpy() - R["mulaw_tensor_f32"]).max() <= 2 ** -23
    y = torch.from_numpy(R["mulaw_tensor_f32"]).cuda()
    assert np.abs(t2.audio.inv_mulaw(y).cpu().numpy() - R["inv_mulaw_tensor_f32"]).max() <= 2e-7
    q = torch.arange(256, dtype=torch.int32).cuda()
    assert np.abs(t2.audio.inv_mulaw_quantize(q).cpu().numpy() - R["inv_mulaw_q_tensor_all"]).max() <= 2e-7
    x64 = torch.from_numpy(R["mulaw_x64"].astype(np.float32)).cuda()       # float64 reference inputs that survive the float32 cast
    safe = np.abs(np.abs((R["mulaw_f64"] + 1) / 2 * 255 % 1.0 - 0.5) - 0.5) > 1e-4     # not within 1e-4 of a bin edge
    assert np.array_equal(t2.audio.mulaw_quantize(x64).cpu().numpy()[safe], R["mulaw_q_f64"][safe])


# ------------------------------------------------------------------------------------------------ datasets/audio.py
def test_oracle_audio_helpers_match_reference():
    from oracle import audio as oa
    hp = hparams.copy()
    assert np.abs(oa.preemphasis(R["wav"], hp.preemphasis, hp.preemphasize) - R["preemphasis"]).max() < 1e-15
    assert np.abs(oa.inv_preemphasis(R["preemphasis"], hp.preemphasis, hp.preemphasize) - R["inv_preemphasis"]).max() < 1e-12
    assert np.abs(oa._amp_to_db(R["S_amp"], hp) - R["amp_to_db"]).max() < 1e-12
    for sym in (1, 0):
        for clip in (1, 0):
            hp.symmetric_mels, hp.allow_clipping_in_normalization = bool(sym), bool(clip)
            src = R["S_db"] if clip else np.clip(R["S_db"], hp.min_level_db, 0.0)
            assert np.abs(oa._normalize(src, hp) - R["normalize_sym%d_clip%d" % (sym, clip)]).max() < 1e-12
            assert np.abs(oa._denormalize(R["denorm_in_sym%d_clip%d" % (sym, clip)], hp) - R["denormalize_sym%d_clip%d" % (sym, clip)]).max() < 1e-10
    hp = hparams.copy()
    hop = oa.get_hop_size(hp)
    assert hop == int(R["hop_size"]) == 275
    for n, a, b in zip(R["pad_lens"], R["librosa_pad_lr_1"], R["librosa_pad_lr_2"]):
        assert tuple(oa.librosa_pad_lr(np.zeros(n), hp.n_fft, hop, 1)) == tuple(a)
        assert tuple(oa.librosa_pad_lr(np.zeros(n), hp.n_fft, hop, 2)) == tuple(b)
    assert tuple(oa.start_and_end_indices(R["silence_q"], hp.silence_threshold)) == tuple(R["start_end"])


def test_oracle_mel_composition_matches_reference_glue():
    """the reference's melspectrogram / linearspectrogram code ran as-is on top of substituted librosa.stft / filters.mel"""
    from oracle import audio as oa
    pre = R["preemphasis"]
    assert np.abs(oa.melspectrogram(pre, hparams) - R["mel_composed"]).max() < 1e-5
    assert np.abs(oa.linearspectrogram(pre, hparams)[::16] - R["linear_composed_rows"]).max() < 1e-5


@pytest.mark.gpu
def test_cuda_audio_matches_reference_vectors():
    from t2_import import t2
    wav = torch.from_numpy(R["wav"]).cuda()[None]
    pre = t2.audio.preemphasis(wav, hparams.preemphasis)
    assert np.abs(pre[0].cpu().numpy() - R["preemphasis"]).max() < 2e-7
    fe = t2.audio.MelFrontEnd(hparams)
    mel, lin = fe(torch.from_numpy(R["preemphasis"].astype(np.float32)).cuda()[None], time_major=False, linear=True)
    assert np.abs(mel[0].cpu().numpy() - R["mel_composed"]).max() < 1e-3
    assert np.abs(lin[0].cpu().numpy()[::16] - R["linear_composed_rows"]).max() < 1e-3


# ------------------------------------------------------------------------------------------------ WaveNet losses / samplers
def test_oracle_mixture_loss_matches_reference_code():
    from oracle import wavenet as ow
    yh, y = torch.from_numpy(R["mol_yhat"]), torch.from_numpy(R["mol_y"])
    lsm = float(np.log(1e-14))
    for nc in (65536, 256):
        ref = R["mol_loss_nc%d" % nc]
        got = ow.discretized_mix_logistic_loss(yh, y, num_classes=nc, log_scale_min=lsm, reduce=False).numpy()
        assert np.abs(got - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), nc
    got = ow.discretized_mix_logistic_loss(yh, y, num_classes=65536, log_scale_min=-7.0, reduce=False).numpy()
    assert np.abs(got - R["mol_loss_lsm7"]).max() <= 1e-5 * np.abs(R["mol_loss_lsm7"]).max()
    assert abs(float(ow.discretized_mix_logistic_loss(yh, y, 65536, lsm, True)) - float(R["mol_loss_sum"])) <= 1e-5 * abs(float(R["mol_loss_sum"]))
    # every branch of the piecewise log-probability is present in the vector
    assert (R["mol_y"] < -0.999).any() and (R["mol_y"] > 0.999).any()
    hp = hparams.copy()
    hp.parse("input_type=raw,quantize_channels=65536,out_channels=30")
    hp.log_scale_min = lsm
    got = ow.masked_mol_loss(yh, y[:, :, 0], torch.from_numpy(R["mol_lengths"]), hp)
    assert abs(float(got) - float(R["mol_add_loss"])) <= 1e-5 * abs(float(R["mol_add_loss"]))
    s = ow.sample_from_discretized_mix_logistic(yh, lsm, torch.from_numpy(R["mol_u_mix"]), torch.from_numpy(R["mol_u_logistic"]))
    assert np.abs(s.numpy() - R["mol_sample"]).max() <= 1e-6


def test_oracle_gaussian_head_matches_reference_code():
    from oracle import wavenet as ow
    gh, y = torch.from_numpy(R["gauss_yhat"]), torch.from_numpy(R["mol_y"])
    for use_cdf in (1, 0):
        got = ow.gaussian_maximum_likelihood_estimation_loss(gh, y, -7.0, 65536, use_cdf=bool(use_cdf), reduce=False).numpy()
        ref = R["gauss_loss_cdf%d" % use_cdf]
        assert np.abs(got - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), use_cdf
    hp = hparams.copy()
    hp.parse("input_type=raw,quantize_channels=65536,out_channels=2,log_scale_min_gauss=-7.0,cdf_loss=False")
    lens = torch.from_numpy(R["mol_lengths"])
    assert abs(float(ow.masked_gaussian_loss(gh, y[:, :, 0], lens, hp)) - float(R["gauss_add_loss"])) <= 1e-5 * abs(float(R["gauss_add_loss"]))
    hp.cdf_loss = True
    assert abs(float(ow.masked_gaussian_loss(gh, y[:, :, 0], lens, hp)) - float(R["gauss_add_loss_cdf"])) <= 1e-5 * abs(float(R["gauss_add_loss_cdf"]))
    s = ow.sample_from_gaussian(gh, -7.0, torch.from_numpy(R["gauss_normal"]))
    assert np.abs(s.numpy() - R["gauss_sample"]).max() <= 1e-6


def test_oracle_masked_cross_entropy_matches_reference_code():
    from oracle import wavenet as ow
    logits, tg = torch.from_numpy(R["ce_logits"]), torch.from_numpy(R["ce_targets"]).long()
    got = ow.masked_cross_entropy(logits.transpose(1, 2), tg, torch.from_numpy(R["ce_lengths"]))
    assert abs(float(got) - float(R["ce_add_loss"])) <= 1e-5 * float(R["ce_add_loss"])
    assert float(R["ce_add_loss"]) != float(R["ce_masked"])           # the shift by one sample matters in the vector


def test_oracle_spectrogram_inversion_matches_reference_code():
    """inv_linear_spectrogram / inv_mel_spectrogram / _griffin_lim of the reference (datasets/audio.py:97-161) executed from its source
    with seeded np.random phases (librosa.stft / istft substituted by the restatements): the oracle reproduces the waveform from the same
    initial phases; the product's pure-numpy helpers agree with the reference's too."""
    from oracle import audio as oa
    it = int(R["gl_iters"])
    ang = np.exp(2j * np.pi * R["gl_u"])
    for key, fn, src in (("gl_wav_from_linear", oa.inv_linear_spectrogram, "gl_linear_in"), ("gl_wav_from_mel", oa.inv_mel_spectrogram, "gl_mel_in")):
        got = fn(R[src], hparams, ang, iters=it)
        ref = R[key]
        assert got.shape == ref.shape
        assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max(), key          # float32 istft outputs, float64 everywhere else
    from datasets import audio as pa
    for sym in (0, 1):
        for clip in (0, 1):
            hp = hparams.copy()
            hp.parse("symmetric_mels=%s,allow_clipping_in_normalization=%s" % (bool(sym), bool(clip)))
            assert np.abs(pa._denormalize(R["denorm_in_sym%d_clip%d" % (sym, clip)], hp) - R["denormalize_sym%d_clip%d" % (sym, clip)]).max() < 1e-12
    assert np.abs(pa._db_to_amp(R["amp_to_db"]) - R["db_to_amp"]).max() <= 1e-12 * np.abs(R["db_to_amp"]).max()


def test_learning_rate_schedules_match_reference_code():
    """Tacotron._learning_rate_decay (tacotron.py:439-463) and WaveNet's noam / exponential schedules (wavenet.py:615-633) executed from
    the reference's classes: the oracle's and the PRODUCT's host-side schedules (engine.learning_rate()) give the same values"""
    from oracle import tacotron as ot, wavenet as ow
    from t2_import import t2
    steps = R["lr_steps"]

    class Eng(object):                       # the engines' learning_rate() only reads self.hp and self.global_step
        pass
    for key, sched, oracle_fn, cls in (("lr_tacotron", None, ot.learning_rate, t2.tacotron.Tacotron),
                                       ("lr_wavenet_noam", "noam", ow.learning_rate, t2.wavenet.WaveNet),
                                       ("lr_wavenet_exponential", "exponential", ow.learning_rate, t2.wavenet.WaveNet)):
        hp = hparams.copy()
        if sched:
            hp.parse("wavenet_lr_schedule=%s" % sched)
        e = Eng()
        e.hp = hp
        for s_, ref in zip(steps, R[key]):
            e.global_step = int(s_)
            assert abs(oracle_fn(hp, int(s_)) - ref) <= 2e-6 * ref, (key, s_)          # float32 pow in the TF op
            assert abs(cls.learning_rate(e) - ref) <= 2e-6 * ref, (key, s_)


# ------------------------------------------------------------------------------------------------ Tacotron pieces
def test_oracle_masked_tacotron_losses_match_reference_code():
    from oracle import tacotron as ot
    tl = torch.from_numpy(R["taco_lengths"]).long()
    got = ot.masked_mse(torch.from_numpy(R["taco_mel_t"]), torch.from_numpy(R["taco_mel_o"]), tl)
    assert abs(float(got) - float(R["taco_masked_mse"])) <= 1e-5 * float(R["taco_masked_mse"])
    got = ot.masked_sigmoid_cross_entropy(torch.from_numpy(R["taco_stop_t"]), torch.from_numpy(R["taco_stop_o"]), tl, float(R["taco_pos_weight"]))
    assert abs(float(got) - float(R["taco_masked_sigmoid_ce"])) <= 1e-5 * float(R["taco_masked_sigmoid_ce"])


def test_oracle_masked_linear_loss_matches_reference_code():
    """MaskedLinearLoss (tacotron/models/modules.py:457-485) executed from the reference's source: L1 with half of the weight on the
    bins below 2 kHz, BOTH terms divided by sum(mask) - the loss of the CBHG linear head when mask_decoder is on"""
    from hparams import hparams
    from oracle import tacotron as ot
    hp = hparams.copy()
    hp.parse("mask_decoder=True")
    got = ot.linear_loss(torch.from_numpy(R["taco_lin_t"]), torch.from_numpy(R["taco_lin_o"]), hp, torch.from_numpy(R["taco_lin_lengths"]).long())
    assert abs(float(got) - float(R["taco_masked_linear"])) <= 1e-5 * float(R["taco_masked_linear"])


def test_oracle_attention_score_matches_reference_code():
    from oracle import tacotron as ot
    wq, wf, wk = (torch.from_numpy(R[k]) for k in ("att_wq", "att_wf", "att_wk"))
    e = ot.location_sensitive_score(wq, wf, wk, torch.from_numpy(R["att_v"]), torch.from_numpy(R["att_b"]))
    assert np.abs(e.numpy() - R["att_score"]).max() <= 2e-5
