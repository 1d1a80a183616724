"""The WaveNet oracle against the reference's OWN graph code, executed: tests/golden/reference_wavenet_graph.npz holds what
`WaveNet(hparams, init).initialize(y, c, g, input_lengths, x=x)` + `add_loss()` of /root/reference/wavenet_vocoder/models/wavenet.py
produce when they run (with modules.py, mixture.py, gaussian.py, util.py underneath) on the TF-1 stand-in of tests/golden/tf_shim*.py
(make_reference_wavenet_graph_vectors.py; the conv primitives there restate TF 1.x, the composition above them is the reference's).
Three scenarios: mu-law cross entropy + SubPixel upsampling, mixture of logistics + ConvTranspose2D, single Gaussian + NearestNeighbor.
Checked here, on CPU: variable names == t2_tf_bundle.wavenet_tf_name over the parameter table; oracle.step / loss_fn reproduce the
network output, the upsampled conditioning and the loss with the recorded dropout masks; d loss / d variable through the oracle ==
autograd through the executed reference graph; the NN_init kernels the reference's `_init_kernel` hands to its upsampling layers ==
the oracle's and the product initialiser's."""
import importlib
import json
import os

import numpy as np
import pytest
import torch

import t2_tf_bundle
from hparams import hparams
from oracle import wavenet as ow

PATH = os.path.join(os.path.dirname(__file__), "golden", "reference_wavenet_graph.npz")
TAGS = ["ce_subpixel", "mol_2d", "gauss_nn", "gauss_paper_2d", "ce_resize", "ce_1d", "mol_gin"]
SUPPORTED = ["ce_subpixel", "mol_2d", "gauss_nn", "gauss_paper_2d"]          # configurations the CUDA path accepts; the rest is oracle only


class _Arrays(dict):
    """name -> array like np.load's NpzFile: `files` lists the names and every lookup returns a fresh copy"""
    @property
    def files(self):
        return list(self)

    def __getitem__(self, name):
        return dict.__getitem__(self, name).copy()


@pytest.fixture(scope="module")
def R():
    """the generator's save_packed() layout: numeric arrays concatenated per dtype, located through `packed_index`"""
    z = np.load(PATH)
    groups = {k: z[k] for k in z.files if k.startswith("packed_") and k != "packed_index"}
    out = _Arrays((k, z[k]) for k in z.files if not k.startswith("packed_"))
    for name, key, off, shape in json.loads(str(z["packed_index"])):
        out[name] = groups["packed_" + key][off:off + int(np.prod(shape, dtype=np.int64))].reshape(shape)
    return out


def _hp(R, tag):
    hp = hparams.copy()
    for keys, values in (("small_hparams_keys", "small_hparams_values"), (tag + "_hparams_keys", tag + "_hparams_values")):
        for k, v in zip(R[keys], R[values]):
            setattr(hp, str(k), eval(str(v)))
    return hp


def _eng(name):
    """reference variable name -> oracle / engine name (the speaker embedding is created outside the `inference` scope, modules.py:12-21)"""
    name = str(name)
    return "gc_embedding" if name == "gc_embedding" else t2_tf_bundle.engine_name("WaveNet_model/" + name)


def _params(R, tag, hp):
    out = {}
    for name in R[tag + "_var_names"]:
        eng = _eng(name)
        assert eng is not None, name
        out[eng] = torch.from_numpy(R["%s_var/%s" % (tag, name)]).clone().requires_grad_(True)
    return out


@pytest.mark.parametrize("tag", TAGS)
def test_variable_names_match_the_checkpoint_name_map(R, tag):
    hp = _hp(R, tag)
    got = {"WaveNet_model/" + str(n): tuple(R["%s_var/%s" % (tag, n)].shape) for n in R[tag + "_var_names"]}
    want = {("WaveNet_model/gc_embedding" if k == "gc_embedding" else t2_tf_bundle.wavenet_tf_name(k, hp.upsample_type)): tuple(v)
            for k, v in ow.param_shapes(hp).items()}
    assert set(got) == set(want), (sorted(set(got) - set(want))[:4], sorted(set(want) - set(got))[:4])
    assert got == want


@pytest.mark.parametrize("tag", TAGS)
def test_training_graph_output_loss_and_gradients(R, tag):
    hp = _hp(R, tag)
    params = _params(R, tag, hp)
    x, c = torch.from_numpy(R[tag + "_x"]), torch.from_numpy(R["c"])
    lengths = torch.from_numpy(R["input_lengths"]).long()
    masks = [torch.from_numpy(R["%s_mask_%d" % (tag, l)]) for l in range(hp.layers)]
    up = ow.upsample(c, params, hp)
    assert np.abs(up.detach().numpy() - R[tag + "_upsampled_c"]).max() <= 2e-6
    g = torch.from_numpy(R[tag + "_g"]) if tag + "_g" in R.files else None
    y_hat = ow.step(x, c, params, hp, dropout_masks=masks, g=g)
    ref = R[tag + "_y_hat"]
    assert y_hat.shape == ref.shape and np.abs(y_hat.detach().numpy() - ref).max() <= 2e-5 * max(1.0, np.abs(ref).max())
    y = torch.from_numpy(R[tag + "_y"])[:, :, 0]
    y = y.long() if ow.is_mulaw_quantize(hp.input_type) else y
    loss = ow.loss_fn(y_hat, y, lengths, hp)
    assert abs(float(loss.detach()) - float(R[tag + "_loss"])) <= 1e-5 * abs(float(R[tag + "_loss"]))
    loss.backward()
    floor = 1e-3 * max(np.abs(R[k]).max() for k in R.files if k.startswith(tag + "_grad/"))
    for name in R[tag + "_var_names"]:
        eng = _eng(name)
        ref = R["%s_grad/%s" % (tag, name)]
        g = params[eng].grad
        g = np.zeros_like(ref) if g is None else g.numpy()
        assert np.abs(g - ref).max() <= 2e-4 * max(np.abs(ref).max(), floor), eng


@pytest.mark.parametrize("tag", ["ce_subpixel", "mol_2d", "ce_resize", "ce_1d"])
def test_nn_init_kernels_of_the_reference_match_oracle_and_product_initialisers(R, tag):
    hp = _hp(R, tag)
    init = importlib.import_module("tacotron-2_b200.init")
    keys = [k for k in R.files if k.startswith(tag + "_init/")]
    assert len(keys) == len(hp.upsample_scales)
    for k in keys:
        eng = t2_tf_bundle.engine_name("WaveNet_model/" + k.split("/", 1)[1])            # local_conditioning_upsampling_<i>/kernel
        i = int(eng.split("/")[0].rsplit("_", 1)[1]) - 1
        shape = ow.param_shapes(hp)[eng]
        ref = R[k].reshape(shape)         # tf.constant_initializer fills the variable in row-major order (see the generator's note)
        assert np.abs(ow._upsample_init_kernel(hp, i, hp.upsample_scales[i]).numpy() - ref).max() <= 1e-7
        if tag in SUPPORTED:
            prod = init.nn_upsample_kernel(shape, hp.upsample_scales[i], len(hp.upsample_scales), hp.NN_scaler, hp.upsample_type == "SubPixel")
            assert np.abs(prod.numpy() - ref).max() <= 1e-7
        assert float(np.abs(ref).sum()) > 0


def _plain_params(R, tag):
    return {_eng(n): torch.from_numpy(R["%s_var/%s" % (tag, n)]) for n in R[tag + "_var_names"]}


AR_TAGS = ["ce_subpixel", "mol_2d", "gauss_nn", "gauss_paper_2d"]


@pytest.mark.parametrize("tag", AR_TAGS)
def test_evaluation_branch_teacher_forced_incremental_pass(R, tag):
    """wavenet.py:382-440 + incremental (:724-911): item 0, Fast-WaveNet queues, next input = the ground-truth sample; the raw network
    outputs of the incremental pass equal the oracle's incremental AND its parallel forward; eval loss (:497-507) restated here"""
    hp = _hp(R, tag)
    params = _plain_params(R, tag)
    n = int(R[tag + "_eval_length"])
    c0 = torch.from_numpy(R["c"])[:1]
    y0 = torch.from_numpy(R[tag + "_y"])[:1, :n]                                       # [1, T, 1]
    if ow.is_mulaw_quantize(hp.input_type):
        Q = hp.quantize_channels
        test_inputs = torch.nn.functional.one_hot(y0[:, :, 0].long(), Q).float()
        initial = torch.nn.functional.one_hot(torch.tensor([[127]]), Q).float()          # mulaw_quantize(0) (util.py:71-102)
    else:
        test_inputs, initial = y0, torch.zeros(1, 1, 1)
    outs, raws = ow.incremental(initial, c0, params, hp, n, test_inputs=test_inputs, u_cat=torch.full((1, n), 0.5),
                                u_mix=torch.full((1, n, max(hp.out_channels // 3, 1)), 0.5), u_logistic=torch.full((1, n), 0.5),
                                normal=torch.zeros(1, n))
    ref = torch.from_numpy(R[tag + "_eval_raw"])
    ref = ref if ow.is_mulaw_quantize(hp.input_type) else ref.transpose(1, 2)         # -> [1, T, out]
    assert (raws - ref).abs().max() <= 2e-5 * max(1.0, float(ref.abs().max()))
    x_par = torch.cat([initial, test_inputs[:, :-1]], dim=1).transpose(1, 2)           # the same inputs, as one parallel pass
    par = ow.step(x_par, c0, params, hp).transpose(1, 2)
    assert (par - ref).abs().max() <= 5e-5 * max(1.0, float(ref.abs().max()))
    if ow.is_mulaw_quantize(hp.input_type):
        loss = torch.nn.functional.cross_entropy(ref[0], y0[0, :, 0].long())
    elif hp.out_channels == 2:
        loss = ow.gaussian_maximum_likelihood_estimation_loss(ref.transpose(1, 2), y0, hp.log_scale_min_gauss, hp.quantize_channels,
                                                              use_cdf=hp.cdf_loss, reduce=False).mean()
    else:
        loss = ow.discretized_mix_logistic_loss(ref.transpose(1, 2), y0, num_classes=hp.quantize_channels, log_scale_min=hp.log_scale_min,
                                                reduce=False).mean()
    assert abs(float(loss) - float(R[tag + "_eval_loss"])) <= 2e-5 * abs(float(R[tag + "_eval_loss"]))


@pytest.mark.parametrize("tag", AR_TAGS)
def test_synthesis_branch_free_running_with_the_recorded_draws(R, tag):
    """wavenet.py:441-478: conditioning [B, Tc, cin] in, Tc * hop samples out; every categorical / mixture / logistic draw of the
    executed reference is injected into the oracle, so the sampled waveforms must agree sample by sample"""
    from oracle import audio as oa
    hp = _hp(R, tag)
    params = _plain_params(R, tag)
    c = torch.from_numpy(R["c"])
    B, T = c.shape[0], c.shape[2] * hp.hop_size
    if ow.is_mulaw_quantize(hp.input_type):
        Q = hp.quantize_channels
        initial = torch.nn.functional.one_hot(torch.full((B, 1), 127), Q).float()
        outs, raws = ow.incremental(initial, c, params, hp, T, u_cat=torch.from_numpy(R[tag + "_synth_u_cat"]))
        ref_raw = torch.from_numpy(R[tag + "_synth_raw"])                              # [B, T, Q]
        wav = oa.inv_mulaw_quantize(outs.argmax(-1).numpy(), Q)
    elif hp.out_channels == 2:
        outs, raws = ow.incremental(torch.zeros(B, 1, 1), c, params, hp, T, normal=torch.from_numpy(R[tag + "_synth_normal"]))
        ref_raw = torch.from_numpy(R[tag + "_synth_raw"]).transpose(1, 2)
        wav = outs.numpy().reshape(B, T)
    else:
        outs, raws = ow.incremental(torch.zeros(B, 1, 1), c, params, hp, T, u_mix=torch.from_numpy(R[tag + "_synth_u_mix"]),
                                    u_logistic=torch.from_numpy(R[tag + "_synth_u_logistic"]))
        ref_raw = torch.from_numpy(R[tag + "_synth_raw"]).transpose(1, 2)
        wav = outs.numpy().reshape(B, T)
    assert (raws - ref_raw).abs().max() <= 5e-5 * max(1.0, float(ref_raw.abs().max()))
    ref = R[tag + "_synth_y_hat"]
    assert wav.shape == ref.shape == (B, T) and np.abs(wav - ref).max() <= 2e-5
    assert np.unique(np.round(ref, 4)).size > T // 2                                   # a real sampled sequence, not a constant


@pytest.mark.parametrize("tag", TAGS)
def test_one_optimizer_step_of_the_executed_reference(R, tag):
    """wavenet.py:522-633 executed: LR schedule at step 30000, clip_by_norm(100) + clip_by_value(5) per tensor, Adam, then the EMA
    of the UPDATED variables (decay 0.9999). oracle.train_step + adam_step land on the same variables and shadows."""
    hp = _hp(R, tag)
    params = {k: v.detach().clone() for k, v in _plain_params(R, tag).items()}
    x, c = torch.from_numpy(R[tag + "_x"]), torch.from_numpy(R["c"])
    lengths = torch.from_numpy(R["input_lengths"]).long()
    masks = [torch.from_numpy(R["%s_mask_%d" % (tag, l)]) for l in range(hp.layers)]
    y = torch.from_numpy(R[tag + "_y"])[:, :, 0]
    y = y.long() if ow.is_mulaw_quantize(hp.input_type) else y
    step = int(R[tag + "_global_step"])
    assert abs(ow.learning_rate(hp, step) - float(R[tag + "_learning_rate"])) <= 1e-6 * float(R[tag + "_learning_rate"])
    if tag + "_g" in R.files:
        pytest.skip("train_step has no speaker-id argument; the forward / gradient test covers this configuration")
    loss, grads, _ = ow.train_step(params, x, c, y, lengths, hp, dropout_masks=masks)
    new, state = {k: v.clone() for k, v in params.items()}, {}
    lr = ow.adam_step(new, grads, state, hp, step)
    for name in R[tag + "_var_names"]:
        eng = _eng(name)
        old = R["%s_var/%s" % (tag, name)]
        key = "%s_new/%s" % (tag, name)
        if key not in R.files:          # a variable the loss does not reach (the last block's residual output conv): TF hands back a None
            assert eng.startswith("ResidualConv1DGLU_%d/residual_block_out_conv" % (hp.layers - 1)) and float(grads[eng].abs().max()) == 0.0
            delta_ref = np.zeros_like(old)                                       # gradient, the reference skips it (wavenet.py:566-576)
        else:
            delta_ref = R[key] - old
        delta = new[eng].numpy() - params[eng].numpy()
        # measured against the learning rate: Adam's first step is lr * g / (|g| + eps), arbitrary where g is rounding noise around eps
        tol = 5e-3 * lr + 2e-7 * np.abs(old).max()
        assert np.abs(delta - delta_ref).max() <= tol, eng
        ema_ref = R["%s_ema/%s" % (tag, name)] - old
        ema = state["ema"][eng].numpy() - params[eng].numpy()
        assert np.abs(ema - ema_ref).max() <= (1 - hp.wavenet_ema_decay) * tol + 1.2e-7 * np.abs(old).max(), eng
