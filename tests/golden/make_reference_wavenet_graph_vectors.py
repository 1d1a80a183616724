"""Generates tests/golden/reference_wavenet_graph.npz by EXECUTING the reference's own WaveNet graph-construction code
(/root/reference/wavenet_vocoder/models/wavenet.py `WaveNet.__init__` / `initialize` (training branch: `step`) / `add_loss`, with
modules.py - CausalConv1D, Conv1D1x1, ResidualConv1DGLU, SubPixelConvolution, ConvTranspose2D, NearestNeighborUpsample, the masked
losses - mixture.py, gaussian.py and util.py underneath) on the TF-1 stand-in of tf_shim.py + tf_shim_graph.py.

  python tests/golden/make_reference_wavenet_graph_vectors.py        # needs /root/reference; only the committed .npz travels

Scenarios (small widths; every hparam not listed keeps the reference's default - legacy / residual_legacy scaling, dropout 0.05, ...):
  ce_subpixel   input_type mulaw-quantize (256 classes), SubPixel conditioning upsampling, masked cross entropy
  mol_2d        input_type raw, 2-component mixture-of-logistics head, ConvTranspose2D upsampling
  gauss_nn      input_type raw, single-Gaussian head (out_channels 2, the reference default), NearestNeighbor upsampling
  ce_resize / ce_1d / mol_gin  oracle-only variants: ResizeConvolution and ConvTranspose1D upsamplers, global (speaker) conditioning
  gauss_paper_2d  the paper configuration's flags: legacy / residual_legacy off, cdf_loss on, ConvTranspose2D upsampling
Each stores the variables under the names the reference's scopes give them, the recorded dropout masks, the network output, the
loss and d loss / d variable (autograd through the executed reference graph), plus the NN_init kernels the reference hands to its
upsampling layers (`_init_kernel`, modules.py:642-654,761-770).

Honesty: the layer primitives under the reference's code (tf.layers.Conv1D / Conv2D / Conv2DTranspose, keras Wrapper) are
tf_shim_graph.py's restatement of the TF 1.x definitions; the reference's composition of them is executed unchanged."""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"

SMALL = dict(layers=4, stacks=2, residual_channels=8, gate_channels=16, skip_out_channels=8, kernel_size=3, num_mels=6, cin_channels=6,
             gin_channels=-1, hop_size=6, upsample_scales=[2, 3], freq_axis_kernel_size=3, wavenet_num_gpus=1, split_on_cpu=True,
             wavenet_weight_normalization=False,
             wavenet_ema_decay=0.9)       # 0.9999 would move the shadow by less than fp32 spacing in one step: nothing to compare
SCENARIOS = {
    "ce_subpixel": dict(input_type="mulaw-quantize", quantize_channels=256, out_channels=256, upsample_type="SubPixel"),   # util.py hard-codes mu = 255
    "mol_2d": dict(input_type="raw", quantize_channels=256, out_channels=6, upsample_type="2D"),      # 256 bins: the fp32 cdf difference is not rounding noise
    "gauss_nn": dict(input_type="raw", quantize_channels=65536, out_channels=2, upsample_type="NearestNeighbor"),
    # the flags of the reference's paper configuration (paper_hparams.py:187-195): no sqrt(0.5) scaling of skips / residuals, CDF form
    # of the Gaussian loss with its own log-scale floor (256 bins here: with 65536 the fp32 CDF difference is rounding noise, see mol_2d)
    # variants the product rejects (oracle only): the two other learnable upsamplers and global (speaker) conditioning
    "ce_resize": dict(input_type="mulaw-quantize", quantize_channels=256, out_channels=256, upsample_type="Resize"),
    "ce_1d": dict(input_type="mulaw-quantize", quantize_channels=256, out_channels=256, upsample_type="1D"),
    "mol_gin": dict(input_type="raw", quantize_channels=256, out_channels=6, upsample_type="SubPixel", gin_channels=5, n_speakers=3,
                    use_speaker_embedding=True),
    "gauss_paper_2d": dict(input_type="raw", quantize_channels=256, out_channels=2, upsample_type="2D", legacy=False, residual_legacy=False,
                           cdf_loss=True, log_scale_min_gauss=-7.000000006091266),
}


def save_packed(path, arrays):
    """np.savez_compressed with the numeric arrays of each dtype concatenated into one entry `packed_<dtype>`, located through the
    JSON list `packed_index` of (name, dtype, offset, shape): stored one by one, the ~1450 small arrays of this file would spend a
    third of it on zip headers. tests/test_reference_wavenet_graph.py reads it back."""
    index, groups, sizes, plain = [], {}, {}, {}
    for name in sorted(arrays):
        a = np.asarray(arrays[name])
        if a.dtype.kind not in "biuf":
            plain[name] = a
            continue
        key = a.dtype.name
        index.append((name, key, sizes.get(key, 0), list(a.shape)))
        groups.setdefault(key, []).append(a.reshape(-1))
        sizes[key] = sizes.get(key, 0) + a.size
    np.savez_compressed(path, packed_index=np.array(json.dumps(index)), **plain,
                        **{"packed_" + k: np.concatenate(v) for k, v in groups.items()})


def model_eval_loss(out, tag):
    return out[tag + "_eval_loss"]


def main():
    assert os.path.isdir(REF), "the reference tree is needed to (re)generate these fixtures"
    sys.path.insert(0, HERE)
    import tf_shim
    import tf_shim_graph as G
    G.install()
    # numpy 1.14 (the reference's pin) clipped an out-of-range axis of expand_dims to ndim (with a DeprecationWarning); numpy 2 raises.
    # SubPixelConvolution._init_kernel (modules.py:652) relies on the old behaviour: expand_dims(<2-D>, 3) -> [kh, kw, 1], which
    # np.tile then promotes to [1, kh, kw, filters]; tf.constant_initializer fills the [kh, kw, 1, filters] variable from it in
    # row-major order, i.e. as a reshape.
    _expand = np.expand_dims
    np.expand_dims = lambda a, axis: _expand(a, min(axis, np.ndim(a)) if isinstance(axis, int) and axis >= 0 else axis)
    import keras.utils
    keras.utils.np_utils.to_categorical = lambda y, num_classes=None: np.eye(int(num_classes), dtype=np.float32)[np.asarray(y, dtype=np.int64)]
    sys.path.insert(0, REF)
    import hparams as ref_hparams_mod
    rhp = ref_hparams_mod.hparams
    from wavenet_vocoder.models.wavenet import WaveNet
    Tt = tf_shim.T

    for k, v in SMALL.items():
        assert hasattr(rhp, k), k
        setattr(rhp, k, v)
    out = {"small_hparams_keys": np.array(sorted(SMALL)), "small_hparams_values": np.array([repr(SMALL[k]) for k in sorted(SMALL)])}
    g = torch.Generator().manual_seed(4242)
    B, Tc = 2, 4
    T = Tc * rhp.hop_size
    lengths = torch.tensor([T, T - 7], dtype=torch.int32)
    c = torch.rand(B, rhp.cin_channels, Tc, generator=g)
    out.update(c=c.numpy(), input_lengths=lengths.numpy())

    defaults = {k: getattr(rhp, k) for over in SCENARIOS.values() for k in over}
    for tag, over in SCENARIOS.items():
        for k, v in defaults.items():
            setattr(rhp, k, v)
        for k, v in over.items():
            assert hasattr(rhp, k), k
            setattr(rhp, k, v)
        out[tag + "_hparams_keys"] = np.array(sorted(over))
        out[tag + "_hparams_values"] = np.array([repr(over[k]) for k in sorted(over)])
        if rhp.input_type == "mulaw-quantize":
            q = torch.randint(0, rhp.quantize_channels, (B, T), generator=g)
            x = torch.nn.functional.one_hot(q, rhp.quantize_channels).float().transpose(1, 2)            # [B, classes, T]
            y = q.reshape(B, T, 1).to(torch.int32)
        else:
            wav = torch.rand(B, T, generator=g) * 1.6 - 0.8
            x, y = wav.reshape(B, 1, T), wav.reshape(B, T, 1)
        out[tag + "_x"], out[tag + "_y"] = x.numpy(), y.numpy()

        G.reset(seed=len(tag))
        model = WaveNet(rhp, init=False)
        gids = torch.tensor([[2], [0]], dtype=torch.int32) if rhp.gin_channels > 0 else None
        if gids is not None:
            out[tag + "_g"] = gids.numpy()
        model.initialize(Tt(y.clone()), Tt(c.clone()), None if gids is None else Tt(gids.clone()), Tt(lengths.clone()), x=Tt(x.clone()))
        model.add_loss()
        drops = list(G.S.drops)
        assert len(drops) == rhp.layers and all(k == "layers.dropout" and tuple(m.shape) == (B, rhp.residual_channels, T) for _, k, m in drops), \
            [(s, k, tuple(m.shape)) for s, k, m in drops]
        for l, (scope, _, m) in enumerate(drops):
            assert scope.endswith("ResidualConv1DGLU_%d" % l), scope
            out["%s_mask_%d" % (tag, l)] = (m / (1.0 - rhp.wavenet_dropout)).numpy()
        out[tag + "_y_hat"] = model.tower_y_hat_train[0].detach().numpy()                                  # [B, out_channels, T]
        out[tag + "_upsampled_c"] = model.tower_upsampled_local_features[0].detach().numpy()
        out[tag + "_loss"] = np.asarray(float(model.loss.detach()), dtype=np.float64)
        # one optimizer step (wavenet.py:522-613): LR schedule at global step 30000, per-tensor clip_by_norm + clip_by_value, Adam, EMA
        model.add_optimizer(Tt(torch.tensor(30000)))
        out[tag + "_global_step"] = np.asarray(30000)
        out[tag + "_learning_rate"] = np.asarray(float(model.learning_rate), dtype=np.float64)
        assert model.optimize is model.ema
        for k, v in G.S.assigned.items():
            out["%s_new/%s" % (tag, k)] = v.numpy()
        for k, v in model.ema.shadow.items():
            out["%s_ema/%s" % (tag, k)] = v.numpy()
        model.loss.backward()
        names = list(G.S.vars)
        out[tag + "_var_names"] = np.array(names)
        for k, v in G.S.vars.items():
            out["%s_var/%s" % (tag, k)] = v.detach().numpy()
            out["%s_grad/%s" % (tag, k)] = (v.grad if v.grad is not None else torch.zeros_like(v)).detach().numpy()
        for k, v in G.S.inits.items():
            out["%s_init/%s" % (tag, k)] = v
        print("%s: %d variables, loss %.6f, NN_init kernels recorded: %d" % (tag, len(names), float(model.loss), len(G.S.inits)))
        variables = {k: v.detach().clone() for k, v in G.S.vars.items()}
        if tag not in ("ce_subpixel", "mol_2d", "gauss_nn", "gauss_paper_2d"):
            continue
        cat = rhp.input_type == "mulaw-quantize"

        # ---- evaluation branch (wavenet.py:382-440): item 0, cut to its length, teacher-forced incremental pass + eval loss ------------
        G.reset(seed=100 + len(tag), variables=variables)
        model = WaveNet(rhp, init=False)
        lengths_eval = torch.tensor([T, T - 7], dtype=torch.int32)              # item 0's length must equal Tc * hop (wavenet.py:800 asserts it)
        model.initialize(Tt(y.clone()), Tt(c.clone()), None, Tt(lengths_eval.clone()))
        model.add_loss()
        out[tag + "_eval_length"] = np.asarray(int(lengths_eval[0]))
        out[tag + "_eval_raw"] = model.tower_y_hat_eval[0].detach().numpy()        # CE: [1, T', Q]; MoL: [1, out, T']
        out[tag + "_eval_y_hat"] = model.tower_y_hat[0].detach().numpy()
        out[tag + "_eval_y_target"] = model.tower_y_target[0].detach().numpy()
        out[tag + "_eval_loss"] = np.asarray(float(model.eval_loss.detach()), dtype=np.float64)
        draws = list(G.S.uniforms)
        out[tag + "_eval_n_draws"] = np.asarray(len(draws))
        for i, (kind, u) in enumerate(draws):
            out["%s_eval_draw_%03d" % (tag, i)] = u.detach().numpy()

        # ---- synthesis branch (wavenet.py:441-478): free running from local conditioning [B, Tc, cin], every draw recorded --------------
        G.reset(seed=200 + len(tag), variables=variables)
        model = WaveNet(rhp, init=False)
        model.initialize(None, Tt(c.transpose(1, 2).clone()), None, None)
        out[tag + "_synth_y_hat"] = model.tower_y_hat[0].detach().numpy()          # [B, T] decoded waveform
        out[tag + "_synth_raw"] = model.tower_y_hat_eval[0].detach().numpy()
        draws = list(G.S.uniforms)
        kinds = sorted(set(k for k, _ in draws))
        gauss = rhp.out_channels == 2
        assert len(draws) == (2 * T if not (cat or gauss) else T) and kinds == (["multinomial"] if cat else ["normal"] if gauss else ["random_uniform"]), \
            (len(draws), kinds)
        if gauss:
            out[tag + "_synth_normal"] = torch.cat([u.reshape(B, 1) for _, u in draws], dim=1).numpy()                # [B, T]
        elif cat:
            out[tag + "_synth_u_cat"] = torch.cat([u for _, u in draws], dim=1).numpy()                       # [B, T]
        else:
            out[tag + "_synth_u_mix"] = torch.cat([draws[2 * t][1] for t in range(T)], dim=1).numpy()           # [B, T, nr_mix]
            out[tag + "_synth_u_logistic"] = torch.cat([draws[2 * t + 1][1] for t in range(T)], dim=1).numpy()  # [B, T]
        print("%s: eval loss %.6f over %d samples; synthesis %s" % (tag, float(model_eval_loss(out, tag)), int(lengths_eval[0]),
              out[tag + "_synth_y_hat"].shape))

    path = os.path.join(HERE, "reference_wavenet_graph.npz")
    save_packed(path, out)
    print("wrote %s: %d arrays, %.1f KB" % (path, len(out), os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
