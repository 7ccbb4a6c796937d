"""CPU: pins oracle/e2tts_oracle.py (and the product's host-side mask helpers) against the reference's own e2_tts.py, through
the answers it gave on these cases (tests/golden/reference_cases.npz, minted by oracle/reference_cases.py, which also
describes what is stored and what is redrawn from seeds)."""
import pytest
import torch

from oracle import e2tts_oracle as O
from oracle import reference_cases as R
from conftest import rel_l2

KW = R.KW


@pytest.fixture(scope='module')
def z():
    with R.load() as f:
        return {k: f[k] for k in f.files}


def _forward(z, case, cfg, mel_shape, text, lens, seed, drop_text_cond=False):
    """Oracle forward + backward of stored case `case` (weights and x0 redrawn from the seeds the minting used)."""
    sd = {k: v.requires_grad_(True) for k, v in R.weights(z, case, seed).items()}
    mel = R.randn(mel_shape, 100 + seed)
    o = O.e2tts_forward(sd, cfg, mel, O.list_str_to_tensor(text), lens=torch.tensor(lens) if lens else None,
                        x0=R.randn(mel_shape, 200 + seed), times=torch.from_numpy(z[case + '.times']),
                        span_mask=torch.from_numpy(z[case + '.span_mask']), drop_text_cond=drop_text_cond)
    o['loss'].backward()
    got, want = R.pred_sample(z, case, o['pred'])
    assert rel_l2(got, want) < 1e-4
    return o, {k: v.grad for k, v in sd.items()}


def _loss_close(got, want, rtol):
    got, want = float(torch.as_tensor(got).detach()), float(want)
    assert abs(got - want) <= rtol * abs(want)


@pytest.mark.parametrize('depth,lens', [(2, None), (4, [80, 51])])
def test_forward_backward_vs_reference(z, depth, lens):
    case = f'fwd_d{depth}'
    _, grads = _forward(z, case, O.TransformerCfg(**dict(KW, depth=depth)), (2, 80, 100), ['abc', 'a longer text than the first'], lens, depth)
    R.check_grads(z, case, grads, 2e-4, 1e-7)


def test_melspec_vs_torchaudio(z):
    assert (torch.from_numpy(z['melspec.mel']) - O.melspec(R.randn((1, 256 * 10 + 17), 9))).abs().max() < 1e-3


def test_text_dropped_branch_vs_reference(z):
    """cond_drop (e2_tts.py:1530-1534, :1263-1264): the text stream is skipped, its parameters receive no gradient."""
    o, grads = _forward(z, 'drop', O.TransformerCfg(**dict(KW, heads=4)), (3, 64, 100), ['one', 'two words', ''], [64, 40, 17], 21,
                        drop_text_cond=True)
    _loss_close(o['loss'], z['drop.loss'], 1e-5)
    R.check_grads(z, 'drop', grads, 2e-4, 1e-7, unused_stay_zero=True)


def test_variant_state_dicts_match_reference(z):
    """The non-default switches that are built (attn_fourier_embed_input, interpolated_text, concat_cond) keep the reference's parameter names
    and shapes, so reference checkpoints of those variants load."""
    import e2_tts_pytorch_b200 as pkg
    kw = dict(transformer=dict(dim=128, depth=2, heads=2, attn_fourier_embed_input=True), use_vocos=False, interpolated_text=True,
              concat_cond=True)
    a = {str(k): str(s) for k, s in zip(z['variants.names'], z['variants.shapes'])}
    b = {k: ','.join(str(s) for s in v.shape) for k, v in pkg.E2TTS(**kw).state_dict().items()}
    assert set(a) == set(b), (sorted(set(a) - set(b))[:5], sorted(set(b) - set(a))[:5])
    for k in a:
        assert a[k] == b[k], k


def test_concat_cond_vs_reference(z):
    """E2TTS(concat_cond=True) (e2_tts.py:1134, :1200-1201, :1263-1267): one Linear(2C -> dim) on cat(cond, x) instead of two summed
    projections — the reference's own code."""
    shapes = dict(zip(z['concat.names'], z['concat.shapes']))
    assert 'cond_proj_in.weight' not in shapes and shapes['proj_in.weight'] == '128,200'
    o, grads = _forward(z, 'concat', O.TransformerCfg(**KW), (2, 64, 100), ['abc', 'defgh ij'], [64, 41], 29)
    _loss_close(o['loss'], z['concat.loss'], 1e-5)
    R.check_grads(z, 'concat', grads, 2e-4, 1e-7)


def test_interpolated_text_vs_reference(z):
    """E2TTS(interpolated_text=True) (e2_tts.py:1135, :1233; InterpolatedCharacterEmbed :414-482, interpolate_1d :237-244) — the
    reference's own code: ragged text lengths, ragged audio lengths, loss / prediction / every gradient incl. the embedding table and
    both abs_pos_mlp linears."""
    assert 'embed_text.abs_pos_mlp.3.weight' in set(z['interp.names'])
    o, grads = _forward(z, 'interp', O.TransformerCfg(**KW), (3, 64, 100), ['abc', 'a much longer piece of text', 'xy'], [64, 45, 30], 27)
    _loss_close(o['loss'], z['interp.loss'], 1e-5)
    R.check_grads(z, 'interp', grads, 2e-4, 1e-7)
    assert float(grads['embed_text.abs_pos_mlp.1.weight'].abs().max()) > 0 and float(grads['embed_text.embed.weight'].abs().max()) > 0


def test_attn_fourier_embed_input_vs_reference(z):
    """Transformer(attn_fourier_embed_input=True) (e2_tts.py:545-546, LinearFourierEmbed :368-386 applied at :909) — the reference's own
    code, no third-party leaf involved: loss, prediction and every gradient incl. `layers.{i}.0.4.linear.weight`."""
    assert 'transformer.layers.0.0.4.linear.weight' in set(z['fourier.names'])
    o, grads = _forward(z, 'fourier', O.TransformerCfg(**KW), (2, 64, 100), ['abc', 'defgh ij'], [64, 45], 23)
    _loss_close(o['loss'], z['fourier.loss'], 1e-5)
    R.check_grads(z, 'fourier', grads, 2e-4, 1e-7)
    assert float(grads['transformer.layers.1.0.4.linear.weight'].abs().max()) > 0


@pytest.mark.parametrize('steps,cfg_strength,duration', R.SAMPLE_CASES)
def test_sample_vs_reference(z, steps, cfg_strength, duration):
    """E2TTS.sample (:1332-1466): midpoint grid, CFG with the APG orthogonal projection (:1303-1330, :113-124), the
    cond mask / duration logic (:1376-1405) — same y0 injected into the oracle."""
    i = R.SAMPLE_CASES.index((steps, cfg_strength, duration))
    dur = torch.tensor(duration) if isinstance(duration, list) else duration
    with torch.no_grad():
        got = O.e2tts_sample(R.weights(z, 'sample', 31), O.TransformerCfg(**KW), R.randn((2, 20, 100), 131),
                             O.list_str_to_tensor(['Hello', 'Goodbye then']), duration=dur, y0=R.randn(z[f'sample{i}.y0_shape'], 300 + i),
                             steps=steps, cfg_strength=cfg_strength)
    got, want = R.pred_sample(z, f'sample{i}', got)
    assert rel_l2(got, want) < 1e-4


def test_duration_predictor_vs_reference(z):
    """DurationPredictor.forward (:1042-1113): random prefix mask, masked mean pool, softplus head, L1-on-frames loss."""
    sd = {k: v.requires_grad_(True) for k, v in R.weights(z, 'duration', 41).items()}
    got = O.duration_forward(sd, O.TransformerCfg(cond_on_time=False, **KW), R.randn((3, 72, 100), 141),
                             O.list_str_to_tensor(['abc', 'hello world', 'x']), lens=torch.tensor([72, 50, 31]),
                             rand_frac=torch.from_numpy(z['duration.rand_frac']))
    _loss_close(got, z['duration.loss'], 1e-4)
    got.backward()
    R.check_grads(z, 'duration', {k: v.grad for k, v in sd.items()}, 5e-4, 1e-6)


def test_mask_helpers_bit_exact_vs_reference(z):
    """The product's host-side mask helpers (e2-tts-pytorch_b200/modules.py: lens_to_mask, mask_from_frac_lengths — SURVEY §8 row a14)
    against the reference's (e2_tts.py:173-210), bit for bit on 200 seeded ragged cases (same torch RNG state -> same rand_like draw)."""
    import numpy as np
    import e2_tts_pytorch_b200 as pkg
    want = {k: torch.from_numpy(np.unpackbits(z['masks.' + k]).astype(bool)) for k in ('frac', 'lens_n', 'lens')}
    at = dict.fromkeys(want, 0)

    def check(k, got, case):
        w = want[k][at[k]:at[k] + got.numel()]
        at[k] += got.numel()
        assert got.dtype == torch.bool and torch.equal(got.flatten(), w), (k, case)

    g = torch.Generator().manual_seed(0)
    for case in range(200):
        b = int(torch.randint(1, 9, (1,), generator=g))
        n = int(torch.randint(8, 300, (1,), generator=g))
        lens = torch.randint(1, n + 1, (b,), generator=g)
        if case % 3 == 0:
            lens[int(torch.randint(0, b, (1,), generator=g))] = n
        frac = torch.rand(b, generator=g) * 0.3 + 0.7          # frac_lengths_mask = (0.7, 1.0), e2_tts.py:1133
        torch.manual_seed(1000 + case)
        got = pkg.mask_from_frac_lengths(lens, frac, n)
        assert got.shape == (b, n), case
        check('frac', got, case)
        check('lens_n', pkg.lens_to_mask(lens, length=n), case)
        got = pkg.lens_to_mask(lens)
        assert got.shape == (b, int(lens.max())), case
        check('lens', got, case)
    for k in want:          # every stored bit was compared; packbits pads the last byte with zeros
        assert want[k].numel() - at[k] < 8 and not want[k][at[k]:].any(), k
    ids = pkg.list_str_to_tensor(['Hello', 'Goodbye', 'héllo wörld'])
    assert torch.equal(ids, torch.from_numpy(z['masks.text_ids']))


def test_velocity_consistency_loss_vs_reference(z):
    """E2TTS.forward with a velocity_consistency_model (e2_tts.py:1556-1576, trainer hook trainer.py:259-268): total loss, breakdown and
    gradients of the online model against the oracle's restatement."""
    sd = {k: v.requires_grad_(True) for k, v in R.weights(z, 'velocity', 5).items()}
    o = O.e2tts_forward(sd, O.TransformerCfg(**KW), R.randn((2, 64, 100), 105), O.list_str_to_tensor(['abc', 'some text']),
                        lens=torch.tensor([64, 50]), x0=R.randn((2, 64, 100), 205), times=torch.from_numpy(z['velocity.times']),
                        span_mask=torch.from_numpy(z['velocity.span_mask']), velocity_sd=R.weights(z, 'velocity_ema', 6),
                        velocity_consistency_weight=0.7, velocity_consistency_delta=1e-3)
    o['loss'].backward()
    _loss_close(o['loss'], z['velocity.loss'], 1e-5)
    _loss_close(o['flow_loss'], z['velocity.flow_loss'], 1e-5)
    _loss_close(o['velocity_loss'], z['velocity.velocity_loss'], 1e-5)
    assert float(z['velocity.velocity_loss']) > 0
    # fp32 summation order differs between the two autograd graphs (and with the host's thread count), and the velocity term's finite
    # difference divides by delta = 1e-3, amplifying fp32 rounding ~1000x: norm-wise agreement with an absolute floor of 1e-4 of the
    # total gradient norm (scalar parameters summed over every token sit at 1-3e-5) (measured under host load, where the BLAS thread
    # partition changes: up to 2.5e-3 of a parameter's own gradient norm)
    R.check_grads_norm(z, 'velocity', {k: v.grad for k, v in sd.items()}, 6e-3, 1e-4)
