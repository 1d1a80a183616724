"""Generates tests/golden/reference_exec.npz + reference_hparams.json by EXECUTING the reference's own Python source
(/root/reference, read-only) in this container.

  python tests/golden/make_reference_vectors.py        # needs /root/reference; the GPU box only sees the committed files

What is executed, and how honest each fixture is:
  * numpy code paths (wavenet_vocoder/util.py mu-law family, datasets/audio.py pre-emphasis / dB / normalise / padding
    helpers, feeder padding helpers): the reference's code runs AS IS on numpy 2.3 / scipy 1.18 (the reference pins numpy 1.14:
    under NEP-50 a float32 array divided by the np.float64 scalar np.log1p(255) promotes to float64, which numpy 1.14's
    value-based casting did not do - so the float64 vectors are exact, and the float32 production path is taken from the
    reference's TENSOR code path below, which stays in float32 like numpy 1.14 did);
  * TF tensor code paths (mu-law family on tensors, mixture.py / gaussian.py losses and samplers, the masked losses of
    wavenet_vocoder/models/modules.py and tacotron/models/modules.py, attention.py score functions): the reference's code runs
    AS IS on tests/golden/tf_shim.py, a torch-CPU stand-in that implements only ELEMENTARY ops by their documented TF-1.x
    meaning (exp, sigmoid, softplus, where, reduce_*, one_hot, sequence_mask, ...). Random draws are injected;
  * datasets/audio.py melspectrogram / linearspectrogram: the reference's glue (power, mel matmul, dB, normalise, call
    signatures, hparams values) runs AS IS; the two librosa primitives it calls (librosa.stft, librosa.filters.mel) are NOT
    available and are substituted by the oracle's restatements (cross-checked against torch.stft / torchaudio in
    tests/test_oracle_audio.py). These vectors pin the composition, not the primitives. The same holds for the inversion path
    (inv_linear_spectrogram / inv_mel_spectrogram / _griffin_lim with librosa.istft substituted).
Layers built from tf.layers / tf.nn.rnn_cell / seq2seq (convolutions, LSTM cells, BahdanauAttention) are not executed HERE; the
reference's whole Tacotron graph code runs in make_reference_graph_vectors.py on tf_shim_graph.py's stand-in for those classes."""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"


def _load_oracle_audio():
    import importlib.util
    spec = importlib.util.spec_from_file_location("oracle_audio_for_stub", os.path.join(ROOT, "oracle", "audio.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def main():
    assert os.path.isdir(REF), "the reference tree is needed to (re)generate these fixtures"
    sys.path.insert(0, HERE)
    import tf_shim
    tf = tf_shim.install()
    oa = _load_oracle_audio()
    sys.path.insert(0, REF)
    import hparams as ref_hparams_mod                       # the reference's hparams.py, HParams(**values) captured by the shim
    rhp = ref_hparams_mod.hparams
    from datasets import audio as ra
    from wavenet_vocoder import util as ru
    from wavenet_vocoder.models import mixture as rmix, gaussian as rgauss, modules as rwm
    from tacotron.models import modules as rtm, attention as ratt
    import tacotron.feeder as rtf
    import wavenet_vocoder.feeder as rwf

    out = {}
    rng = np.random.default_rng(20260923)
    g = torch.Generator().manual_seed(20260923)

    # ---------------- hparams: the reference's own default values --------------------------------------------
    hp_json = {k: (list(v) if isinstance(v, tuple) else v) for k, v in sorted(vars(rhp).items())
               if isinstance(v, (int, float, str, bool, list, tuple, type(None)))}
    json.dump(hp_json, open(os.path.join(HERE, "reference_hparams.json"), "w"), indent=1, sort_keys=True)

    # ---------------- A. mu-law family (wavenet_vocoder/util.py:30-129) ------------------------------------------
    edge = np.array([-1.0, -0.999999, -0.5, -1e-3, -1e-7, 0.0, 1e-7, 1e-3, 0.5, 0.999999, 1.0])
    # bin edges of the quantiser, approached from both sides (truncation toward zero decides the index)
    k = np.arange(1, 255, dtype=np.float64)
    y_edge = k / 255.0 * 2 - 1
    x_edge = np.sign(y_edge) * (1.0 / 255) * ((1.0 + 255) ** np.abs(y_edge) - 1.0)
    x64 = np.concatenate([edge, x_edge, np.nextafter(x_edge, 1), np.nextafter(x_edge, -1), rng.uniform(-1, 1, 1000)])
    out["mulaw_x64"] = x64
    out["mulaw_f64"] = ru.mulaw(x64)
    out["mulaw_q_f64"] = ru.mulaw_quantize(x64).astype(np.int32)
    out["inv_mulaw_f64"] = ru.inv_mulaw(out["mulaw_f64"])
    out["inv_mulaw_q_all"] = ru.inv_mulaw_quantize(np.arange(256))                 # numpy path: float32 in, see util.py:127
    x32 = np.concatenate([edge, x_edge, rng.uniform(-1, 1, 2000)]).astype(np.float32)
    xt = torch.from_numpy(x32)
    out["mulaw_x32"] = x32
    out["mulaw_tensor_f32"] = ru.mulaw(xt).numpy()                                     # tensor path: float32 end to end
    out["mulaw_q_tensor_f32"] = ru.mulaw_quantize(xt).numpy().astype(np.int32)         # tf.cast(., int32) truncation (util.py:156)
    out["inv_mulaw_tensor_f32"] = ru.inv_mulaw(torch.from_numpy(out["mulaw_tensor_f32"])).numpy()
    out["inv_mulaw_q_tensor_all"] = ru.inv_mulaw_quantize(torch.arange(256)).numpy()
    out["mulaw_q_numpy_f32_numpy2"] = ru.mulaw_quantize(x32).astype(np.int32)          # numpy-2 promotion path (documentation only)
    out["mulaw_q_scalar0"] = np.array([ru.mulaw_quantize(0), ru.mulaw_quantize(0.0)])
    out["numpy_version"] = np.array(np.__version__)

    # ---------------- B. datasets/audio.py -------------------------------------------------------------------------
    wav = (0.5 * np.sin(np.cumsum(np.linspace(0.01, 0.6, 3000))) + rng.normal(0, 0.05, 3000)).astype(np.float32)
    wav = (wav / np.abs(wav).max() * rhp.rescaling_max).astype(np.float32)
    out["wav"] = wav
    out["preemphasis"] = ra.preemphasis(wav, rhp.preemphasis, rhp.preemphasize)
    out["inv_preemphasis"] = ra.inv_preemphasis(out["preemphasis"], rhp.preemphasis, rhp.preemphasize)
    S = rng.uniform(1e-7, 30.0, (80, 8))
    out["S_amp"] = S
    out["amp_to_db"] = ra._amp_to_db(S, rhp)
    out["db_to_amp"] = ra._db_to_amp(out["amp_to_db"])
    Sdb = rng.uniform(-130.0, 10.0, (80, 8))
    out["S_db"] = Sdb
    for sym in (True, False):
        for clip in (True, False):
            rhp.symmetric_mels, rhp.allow_clipping_in_normalization = sym, clip
            src = Sdb if clip else np.clip(Sdb, rhp.min_level_db, 0.0)     # the un-clipped branch asserts its input range
            out["normalize_sym%d_clip%d" % (sym, clip)] = ra._normalize(src, rhp)
            D = rng.uniform(-5.0, 5.0, (80, 8)) if clip else ra._normalize(src, rhp)
            out["denorm_in_sym%d_clip%d" % (sym, clip)] = D
            out["denormalize_sym%d_clip%d" % (sym, clip)] = ra._denormalize(D, rhp)
    rhp.symmetric_mels, rhp.allow_clipping_in_normalization = True, True
    lens = np.array([1, 274, 275, 276, 1100, 22050, 31234])
    out["pad_lens"] = lens
    out["librosa_pad_lr_1"] = np.array([ra.librosa_pad_lr(np.zeros(n), rhp.n_fft, ra.get_hop_size(rhp), 1) for n in lens])
    out["librosa_pad_lr_2"] = np.array([ra.librosa_pad_lr(np.zeros(n), rhp.n_fft, ra.get_hop_size(rhp), 2) for n in lens])
    out["pad_lr"] = np.array([ra.pad_lr(np.zeros(n), rhp.n_fft, ra.get_hop_size(rhp)) for n in lens])
    out["num_frames"] = np.array([ra.num_frames(n, rhp.n_fft, ra.get_hop_size(rhp)) for n in lens])
    out["hop_size"] = np.array(ra.get_hop_size(rhp))
    q = ru.mulaw_quantize(np.concatenate([np.zeros(300), wav[:2000].astype(np.float64), np.zeros(500)]))
    out["silence_q"] = q.astype(np.int32)
    out["start_end"] = np.array(ra.start_and_end_indices(q, rhp.silence_threshold))
    # composition through the reference's melspectrogram / linearspectrogram with the two librosa primitives substituted
    import librosa
    from types import SimpleNamespace as NS

    def stft_stub(y=None, n_fft=2048, hop_length=None, win_length=None, pad_mode="reflect", **kw):
        assert pad_mode == "constant" and not kw, "the reference calls librosa.stft(y, n_fft, hop_length, win_length, pad_mode='constant')"
        return oa.stft(y, NS(n_fft=n_fft, hop_size=hop_length, win_size=win_length))
    librosa.stft = stft_stub
    librosa.filters.mel = lambda sr, n_fft, n_mels=128, fmin=0.0, fmax=None, **kw: oa.build_mel_basis(
        NS(sample_rate=sr, n_fft=n_fft, num_mels=n_mels, fmin=fmin, fmax=fmax))
    pre = ra.preemphasis(wav, rhp.preemphasis, rhp.preemphasize)
    out["mel_composed"] = ra.melspectrogram(pre, rhp)
    out["linear_composed_rows"] = ra.linearspectrogram(pre, rhp)[::16].astype(np.float32)        # every 16th frequency row
    out["mel_composed"] = out["mel_composed"].astype(np.float32)

    # ---------------- C. mixture of logistics (mixture.py:18-107, modules.py:800-817) ----------------------------------
    B, Tm, nm = 3, 64, 10
    yh = torch.randn(B, 3 * nm, Tm, generator=g)
    yh[:, nm:2 * nm] *= 0.6                                      # means
    yh[:, 2 * nm:] = yh[:, 2 * nm:] * 3.0 - 5.0                  # log-scales down to ~ -14: exercises clamp + the mid-pdf branch
    y = (torch.rand(B, Tm, 1, generator=g) * 2 - 1)
    y[0, :8, 0] = torch.tensor([-1.0, -0.9995, 0.9995, 1.0, -0.999, 0.999, 0.0, 0.5])   # both edge branches
    lsm = float(np.log(1e-14))
    out["mol_yhat"], out["mol_y"] = yh.numpy(), y.numpy()
    for nc in (65536, 256):
        out["mol_loss_nc%d" % nc] = rmix.discretized_mix_logistic_loss(yh, y, num_classes=nc, log_scale_min=lsm, reduce=False).numpy()
    out["mol_loss_sum"] = np.array(float(rmix.discretized_mix_logistic_loss(yh, y, num_classes=65536, log_scale_min=lsm, reduce=True)))
    out["mol_loss_lsm7"] = rmix.discretized_mix_logistic_loss(yh, y, num_classes=65536, log_scale_min=-7.0, reduce=False).numpy()
    mol_lengths = torch.tensor([Tm, 50, 31])
    rhp.quantize_channels, rhp.log_scale_min = 65536, lsm
    out["mol_lengths"] = mol_lengths.numpy()
    out["mol_masked_mean"] = np.array(float(rwm.DiscretizedMixtureLogisticLoss(yh, y, rhp, lengths=mol_lengths, max_len=Tm)))
    # exactly as WaveNet.add_loss composes it (wavenet.py:488-495, get_mask :632-638): shifted by one sample
    from wavenet_vocoder.models.wavenet import WaveNet as RefWaveNet
    from types import SimpleNamespace as NS0
    rhp.input_type = "raw"
    mask_raw = RefWaveNet.get_mask(NS0(_hparams=rhp), mol_lengths, maxlen=Tm)
    out["mol_add_loss"] = np.array(float(rwm.DiscretizedMixtureLogisticLoss(yh[:, :, :-1], y[:, 1:, :], hparams=rhp, mask=mask_raw)))
    u1 = torch.rand(B, Tm, nm, generator=g) * (1 - 2e-5) + 1e-5
    u2 = torch.rand(B, Tm, generator=g) * (1 - 2e-5) + 1e-5
    tf_shim.inject(uniform=[u1, u2])
    out["mol_u_mix"], out["mol_u_logistic"] = u1.numpy(), u2.numpy()
    out["mol_sample"] = rmix.sample_from_discretized_mix_logistic(yh, log_scale_min=lsm).numpy()

    # ---------------- D. single Gaussian head (gaussian.py:5-52, modules.py:819-836) -------------------------------------
    gh = torch.randn(B, 2, Tm, generator=g)
    gh[:, 1] = gh[:, 1] * 2.0 - 4.0
    out["gauss_yhat"] = gh.numpy()
    for use_cdf in (True, False):
        out["gauss_loss_cdf%d" % use_cdf] = rgauss.gaussian_maximum_likelihood_estimation_loss(
            gh, y, log_scale_min_gauss=-7.0, num_classes=65536, use_cdf=use_cdf, reduce=False).numpy()
    rhp.log_scale_min_gauss, rhp.cdf_loss = -7.0, False
    out["gauss_masked_mean"] = np.array(float(rwm.GaussianMaximumLikelihoodEstimation(gh, y, rhp, lengths=mol_lengths, max_len=Tm)))
    out["gauss_add_loss"] = np.array(float(rwm.GaussianMaximumLikelihoodEstimation(gh[:, :, :-1], y[:, 1:, :], hparams=rhp, mask=mask_raw)))
    rhp.cdf_loss = True
    out["gauss_add_loss_cdf"] = np.array(float(rwm.GaussianMaximumLikelihoodEstimation(gh[:, :, :-1], y[:, 1:, :], hparams=rhp, mask=mask_raw)))
    rhp.cdf_loss = False
    nrm = torch.randn(B, Tm, generator=g)
    tf_shim.inject(normal=[nrm])
    out["gauss_normal"] = nrm.numpy()
    out["gauss_sample"] = rgauss.sample_from_gaussian(gh, log_scale_min_gauss=-7.0).numpy()

    # ---------------- E. masked softmax cross entropy (modules.py:781-798) ------------------------------------------------
    Tc_ = 9
    logits = torch.randn(B, Tc_, 256, generator=g) * 3
    tg = torch.randint(0, 256, (B, Tc_), generator=g)
    ce_lengths = torch.tensor([Tc_, 7, 3])
    out["ce_lengths"] = ce_lengths.numpy()
    logits[1, 5] = -80.0
    logits[1, 5, tg[1, 5]] = 80.0                                   # an exactly-zero loss term inside the mask: count_nonzero skips it
    out["ce_logits"], out["ce_targets"] = logits.numpy(), tg.numpy().astype(np.int32)
    out["ce_masked"] = np.array(float(rwm.MaskedCrossEntropyLoss(logits, tg, lengths=ce_lengths, max_len=Tc_)))
    rhp.input_type = "mulaw-quantize"
    mask_q = RefWaveNet.get_mask(NS0(_hparams=rhp), ce_lengths, maxlen=Tc_)
    out["ce_add_loss"] = np.array(float(rwm.MaskedCrossEntropyLoss(logits[:, :-1, :], tg[:, 1:], mask=mask_q)))
    rhp.input_type = "raw"

    # ---------------- F. Tacotron masked losses + attention scores (tacotron/models/modules.py:400-485, attention.py:38-92) --
    Bt, To, M = 3, 16, 80
    tl = torch.tensor([16, 13, 7])
    mt, mo = torch.randn(Bt, To, M, generator=g), torch.randn(Bt, To, M, generator=g)
    st = (torch.arange(To)[None, :] >= (tl[:, None] - 1)).float()
    so = torch.randn(Bt, To, generator=g) * 2
    out["taco_lengths"], out["taco_mel_t"], out["taco_mel_o"] = tl.numpy(), mt.numpy(), mo.numpy()
    out["taco_stop_t"], out["taco_stop_o"] = st.numpy(), so.numpy()
    rhp.outputs_per_step = 1
    out["taco_masked_mse"] = np.array(float(rtm.MaskedMSE(mt, mo, tl, rhp)))
    out["taco_masked_sigmoid_ce"] = np.array(float(rtm.MaskedSigmoidCrossEntropy(st, so, tl, rhp)))
    out["taco_pos_weight"] = np.array(float(rhp.cross_entropy_pos_weight))
    lt, lo_ = torch.randn(Bt, To, rhp.num_freq, generator=g)[:, :2], torch.randn(Bt, To, rhp.num_freq, generator=g)[:, :2]
    tl_lin = torch.tensor([2, 2, 1])
    out["taco_lin_lengths"] = tl_lin.numpy()
    out["taco_lin_t"], out["taco_lin_o"] = lt.numpy(), lo_.numpy()
    out["taco_masked_linear"] = np.array(float(rtm.MaskedLinearLoss(lt, lo_, tl_lin, rhp)))
    rhp.outputs_per_step = 3
    out["taco_seqmask_r3"] = rtm.sequence_mask(torch.tensor([40, 33, 7]), 3, False).numpy()
    rhp.outputs_per_step = 1
    A, Ti = 128, 8
    wq, wf, wk = torch.randn(Bt, 1, A, generator=g), torch.randn(Bt, Ti, A, generator=g), torch.randn(Bt, Ti, A, generator=g)
    va, ba = torch.randn(A, generator=g) * 0.2, torch.randn(A, generator=g) * 0.1
    tf_shim.inject(vars={"attention_variable_projection": va, "attention_bias": ba})
    out["att_wq"], out["att_wf"], out["att_wk"], out["att_v"], out["att_b"] = (t.numpy() for t in (wq, wf, wk, va, ba))
    out["att_score"] = ratt._location_sensitive_score(tf_shim.T(wq), tf_shim.T(wf), tf_shim.T(wk)).numpy()
    out["att_smoothing"] = ratt._smoothing_normalization(torch.from_numpy(np.asarray(out["att_score"]))).numpy()

    # ---------------- G. feeder padding helpers (tacotron/feeder.py:231-256, wavenet_vocoder/feeder.py) ---------------------
    fd = rtf.Feeder.__new__(rtf.Feeder)
    fd._pad, fd._token_pad = 0, 1.0
    fd._target_pad = -(rhp.max_abs_value + 0.1) if rhp.symmetric_mels else -0.1
    out["taco_target_pad"] = np.array(fd._target_pad)
    xi = np.arange(1, 8, dtype=np.int32)
    out["feeder_pad_input"] = fd._pad_input(xi, 10)
    tm_ = rng.normal(size=(7, 4)).astype(np.float32)
    out["feeder_target_in"] = tm_
    out["feeder_pad_target"] = fd._pad_target(tm_, 9)
    out["feeder_pad_token_target"] = fd._pad_token_target(np.zeros(7, dtype=np.float32), 9)
    out["feeder_round_up"] = np.array([fd._round_up(n, 3) for n in range(0, 8)])
    out["feeder_round_down"] = np.array([fd._round_down(n, 3) for n in range(0, 8)])
    out["wn_ensure_divisible"] = np.array([[rwf._ensure_divisible(n, 275, True), rwf._ensure_divisible(n, 275, False)] for n in (274, 275, 276, 8000, 12000)])

    # ---------------- H. spectrogram inversion (datasets/audio.py:97-133 inv_*_spectrogram, :151-161 _griffin_lim) -------------
    # The reference's code runs AS IS (denormalise, dB -> amplitude, magnitude_power / power exponents, pseudo-inverse mel basis, the
    # Griffin-Lim loop with its np.random.rand phases, inverse pre-emphasis); librosa.stft / librosa.istft are substituted by the
    # oracle's restatements like above, and `np.complex` (removed from numpy 1.24) is aliased to the builtin it used to be.
    def istft_stub(D, hop_length=None, win_length=None, **kw):
        assert not kw, "the reference calls librosa.istft(y, hop_length, win_length)"
        return oa.istft(D, NS(n_fft=rhp.n_fft, hop_size=hop_length, win_size=win_length))
    librosa.istft = istft_stub
    if not hasattr(np, "complex"):
        np.complex = complex
    iters_saved = rhp.griffin_lim_iters
    rhp.griffin_lim_iters = 4
    hop = ra.get_hop_size(rhp)
    seg = pre[:hop * 4]
    lin_in = ra.linearspectrogram(seg, rhp).astype(np.float32)           # [1025, 5]
    mel_in = ra.melspectrogram(seg, rhp).astype(np.float32)              # [80, 5]
    out["gl_iters"] = np.array(4)
    out["gl_linear_in"], out["gl_mel_in"] = lin_in, mel_in
    np.random.seed(4321)
    out["gl_u"] = np.random.rand(*lin_in.shape)                          # the draws _griffin_lim makes first (audio.py:155)
    np.random.seed(4321)
    out["gl_wav_from_linear"] = np.asarray(ra.inv_linear_spectrogram(lin_in, rhp), dtype=np.float64)
    np.random.seed(4321)
    out["gl_wav_from_mel"] = np.asarray(ra.inv_mel_spectrogram(mel_in, rhp), dtype=np.float64)
    rhp.griffin_lim_iters = iters_saved

    # ---------------- I. learning-rate schedules (tacotron.py:439-463, wavenet.py:615-633) ---------------------------------------
    # the model classes' own methods, run on instances created without __init__ (only self._hparams is read)
    from tacotron.models import tacotron as rtaco
    from wavenet_vocoder.models import wavenet as rwn
    tm, wm = object.__new__(rtaco.Tacotron), object.__new__(rwn.WaveNet)
    tm._hparams = wm._hparams = rhp
    tm.decay_steps, tm.decay_rate = rhp.tacotron_decay_steps, rhp.tacotron_decay_rate       # set in add_optimizer (tacotron.py:387-388)
    steps = np.array([0, 1, 1000, 3999, 4000, 4001, 20000, 39999, 40000, 50000, 100000, 200000, 310000, 400000, 1000000], dtype=np.int64)
    out["lr_steps"] = steps
    out["lr_tacotron"] = np.array([float(tm._learning_rate_decay(rhp.tacotron_initial_learning_rate, torch.tensor(int(s_)))) for s_ in steps])
    out["lr_wavenet_noam"] = np.array([float(wm._noam_learning_rate_decay(rhp.wavenet_learning_rate, torch.tensor(int(s_)), warmup_steps=rhp.wavenet_warmup))
                                       for s_ in steps])
    out["lr_wavenet_exponential"] = np.array([float(wm._exponential_learning_rate_decay(rhp.wavenet_learning_rate, torch.tensor(int(s_)), rhp.wavenet_decay_rate,
                                                                                         rhp.wavenet_decay_steps)) for s_ in steps])

    # ---------------- J. WaveNet feeder: random hop-aligned crop + conditioning normalisation (wavenet_vocoder/feeder.py:319-401) ---
    wfd = rwf.Feeder.__new__(rwf.Feeder)
    wfd._hparams = rhp
    rj = np.random.RandomState(77)
    hopj = ra.get_hop_size(rhp)
    frames_j = [44, 41, 40, 42]                         # 41+ frames exceed max_time_steps = 11000 (40 frames): those are cropped
    xs = [rj.randint(0, 256, f * hopj).astype(np.int16) for f in frames_j]
    cs_ = [rj.uniform(-4.6, 4.6, (f, 80)).astype(np.float32) for f in frames_j]
    out["wnf_frames"] = np.array(frames_j)
    for i, (x_, c_) in enumerate(zip(xs, cs_)):
        out["wnf_x%d" % i], out["wnf_c%d" % i] = x_, c_
    np.random.seed(2024)
    cropped = wfd._adjust_time_resolution([(x_, c_, 0, len(x_)) for x_, c_ in zip(xs, cs_)], True, wfd._limit_time())
    for i, (x_, c_, _, _) in enumerate(cropped):
        out["wnf_crop_x%d" % i], out["wnf_crop_c%d" % i] = x_, c_
    out["wnf_local_conditions"] = wfd._prepare_local_conditions(True, [b_[1] for b_ in cropped])
    out["wnf_max_time_steps"] = np.array(wfd._limit_time())

    # ---------------- K. Tacotron feeder: one whole batch through the reference's _prepare_batch (tacotron/feeder.py:198-229) ----
    rk = np.random.RandomState(88)
    ex = []
    for i, (nin, nfr) in enumerate([(12, 16), (7, 9), (15, 20), (9, 13)]):
        ex.append((rk.randint(2, 66, nin).astype(np.int32), rk.uniform(-4, 4, (nfr, 80)).astype(np.float32), np.zeros(nfr - 1, dtype=np.float32),
                   rk.uniform(-4, 4, (nfr, 20)).astype(np.float32), nfr))
        out["tf_in%d" % i], out["tf_mel%d" % i], out["tf_lin%d" % i] = ex[-1][0], ex[-1][1], ex[-1][3]
    fd._hparams = rhp
    np.random.seed(99)
    res = fd._prepare_batch(list(ex), 1)
    for name, arr in zip(("inputs", "input_lengths", "mel_targets", "token_targets", "linear_targets", "targets_lengths", "split_infos"), res):
        out["tf_batch_" + name] = arr

    # ---------------- L. Tacotron synthesizer helpers (tacotron/synthesizer.py:236-257): output lengths from the stop tokens ----
    for name in ("pyaudio", "sounddevice"):
        sys.modules.setdefault(name, tf_shim._NoopStub(name))
    from tacotron.synthesizer import Synthesizer as RefTacoSynth
    rl = np.random.default_rng(5)
    stop_rows = rl.random((64, 12)).astype(np.float32)
    stop_rows[0] = 0.1                 # never fires -> the whole row
    stop_rows[1, 0] = 0.9              # fires on the first frame -> length 0
    stop_rows[2, :-1], stop_rows[2, -1] = 0.2, 0.51
    stop_rows[3] = 0.5                 # np.round is half-to-even: 0.5 -> 0, never fires
    out["synth_stop_rows"] = stop_rows
    out["synth_output_lengths"] = np.asarray(RefTacoSynth._get_output_lengths(None, stop_rows))
    rs = RefTacoSynth()
    rs._pad, rs._target_pad = 0, -4.1
    out["synth_pad_input"] = rs._pad_input(np.arange(1, 6, dtype=np.int32), 8)
    out["synth_pad_target"] = rs._pad_target(np.ones((3, 2), dtype=np.float32), 5)
    out["synth_round_up"] = np.asarray([rs._round_up(x, 4) for x in range(0, 10)])

    # ---------------- M. the two preprocessors, one utterance each way (datasets/preprocessor.py:40-165, wavenet_preprocessor.py:39-154) --
    # _process_utterance runs AS IS; substituted underneath: librosa.core.load (scipy wav read -> float32 / 32768, what librosa does for
    # int16 PCM at the native rate), librosa.stft / filters.mel (as in section B), and util._log1p so that a float32 signal stays
    # float32 through mulaw() as it did under numpy 1.14's value-based casting (see this file's header).
    import tempfile
    from scipy.io import wavfile
    import librosa.core
    from datasets import preprocessor as rpre, wavenet_preprocessor as rwpre
    librosa.core.load = lambda path, sr=None, **kw: (wavfile.read(path)[1].astype(np.float32) / 32768.0, sr)
    ru._log1p = lambda x: np.log1p(x) if isinstance(x, np.ndarray) else float(np.log1p(x))
    tmp = tempfile.mkdtemp()
    rm = np.random.default_rng(31337)
    n_m = 3000
    sig = 0.35 * np.sin(np.cumsum(np.linspace(0.02, 0.5, n_m))) * np.hanning(n_m) + 0.004 * rm.standard_normal(n_m)
    sig[:400] = 0.0                                              # leading digital silence: start_and_end_indices has something to cut
    wavfile.write(os.path.join(tmp, "utt.wav"), rhp.sample_rate, (sig * 32767).astype(np.int16))
    out["pre_wav_i16"] = (sig * 32767).astype(np.int16)
    keep = dict(trim_silence=rhp.trim_silence, input_type=rhp.input_type, quantize_channels=rhp.quantize_channels)
    rhp.trim_silence = False
    for itype, qc in (("mulaw-quantize", 256), ("mulaw", 256), ("raw", 65536)):
        rhp.input_type, rhp.quantize_channels = itype, qc
        tag = itype.replace("-", "_")
        d = tempfile.mkdtemp()
        row = rpre._process_utterance(d, d, d, "utt", os.path.join(tmp, "utt.wav"), "some text", rhp)
        out["pre_%s_row" % tag] = np.array([str(x) for x in row])
        out["pre_%s_audio" % tag] = np.load(os.path.join(d, row[0]))
        out["pre_%s_mel" % tag] = np.load(os.path.join(d, row[1]))
        out["pre_%s_linear_cols" % tag] = np.load(os.path.join(d, row[2]))[:, ::16]
        d = tempfile.mkdtemp()
        row = rwpre._process_utterance(d, d, "utt", os.path.join(tmp, "utt.wav"), rhp)
        out["wpre_%s_row" % tag] = np.array([os.path.basename(str(x)) for x in row])
        out["wpre_%s_audio" % tag] = np.load(row[0])
        out["wpre_%s_mel" % tag] = np.load(row[1])
    for k, v in keep.items():
        setattr(rhp, k, v)

    np.savez_compressed(os.path.join(HERE, "reference_exec.npz"), **{k: np.asarray(v) for k, v in out.items()})
    print("wrote %d arrays, %d hparams" % (len(out), len(hp_json)))


if __name__ == "__main__":
    main()
