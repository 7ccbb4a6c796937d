"""The reference's own answers for tests/test_oracle_vs_reference.py, kept in tests/golden/reference_cases.npz.

    python oracle/reference_cases.py     # needs the reference tree (oracle/load_reference.py); rewrites the .npz

Every case runs the reference's e2_tts.py, loaded unmodified, once. Weights and large random inputs are not stored:
  weights  drawn tensor by tensor from a seeded torch.Generator with the mean and standard deviation of the reference's
           own initialisation of that tensor (after O.randomize_zero_init); a constant tensor stays that constant, and a
           tensor of at most EXACT_NUMEL entries (the hyper-connections' 0/1 stream-mixing matrices, gate biases) is kept
           as it is. The file keeps the names, shapes, moments and those small tensors. Buffers the reference computes from its configuration (rotary
           frequencies, STFT window, mel filterbank) are not part of it: the oracle does not read them.
  inputs   mel, cond, wave and the reference's x0 / y0 draws come from seeded generators (`randn`); the small draws
           (times, span masks, the duration prefix fraction) are stored as the reference made them.
  outputs  loss values in full; of each prediction and each parameter gradient a fixed sample of entries
           (`sample_index`) together with the gradient's max-abs and norm, which the tolerances are relative to.
"""
import math
import os
import random
import sys
import zipfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATH = os.path.join(ROOT, 'tests', 'golden', 'reference_cases.npz')
PRED_SAMPLES = 1024       # entries kept of a prediction
GRAD_SAMPLES = 8          # entries kept of each parameter gradient
EXACT_NUMEL = 32          # weight tensors up to this size are stored, not drawn
KW = dict(dim=128, depth=2, heads=2)
SAMPLE_CASES = [(4, 1.0, 48), (3, 0.0, 40), (5, 2.5, [50, 37])]     # E2TTS.sample (steps, cfg_strength, duration)


def sample_index(n, k):
    """k distinct flat indices of an n-element tensor, spread by a prime stride (no RNG: stable across library versions)."""
    return torch.tensor([(j * 1000003) % n for j in range(min(n, k))], dtype=torch.long)


def randn(shape, seed):
    return torch.randn(tuple(shape), generator=torch.Generator().manual_seed(seed))


def load():
    return np.load(PATH, allow_pickle=False)


def weights(z, model, seed):
    """The state dict of stored model `model` (see the module docstring)."""
    g = torch.Generator().manual_seed(seed)
    exact, at = torch.from_numpy(z[model + '.exact']), 0
    sd = {}
    for name, shape, (mean, std) in zip(z[model + '.names'], z[model + '.shapes'], z[model + '.moments'].tolist()):
        shape = tuple(int(s) for s in str(shape).split(',')) if shape else ()
        n = math.prod(shape)
        if std == 0:
            sd[str(name)] = torch.full(shape, mean)
        elif n <= EXACT_NUMEL:
            sd[str(name)] = exact[at:at + n].reshape(shape).clone()
            at += n
        else:
            sd[str(name)] = mean + std * torch.randn(shape, generator=g)
    return sd


def check_grads(z, case, grads, rtol, atol, unused_stay_zero=False):
    """Parameter gradients `grads` ({name: tensor or None}) against the reference's: on the sampled entries and the max-abs,
    |got - want| <= rtol * max|want| + atol, and the norm of the whole gradient within rtol * ||want|| + atol (which catches a
    wrong part of a tensor that the samples miss). With `unused_stay_zero`, a parameter without a gradient in the reference has
    none or an all-zero one here."""
    amax, samples = torch.from_numpy(z[case + '.grad_amax']).double(), torch.from_numpy(z[case + '.grad_samples']).double()
    norm = torch.from_numpy(z[case + '.grad_norm']).double()
    for i, (k, is_param) in enumerate(zip(z[case + '.names'], z[case + '.is_param'])):
        if not is_param:
            continue
        got = grads[str(k)]
        if torch.isnan(amax[i]):      # no gradient in the reference
            assert not unused_stay_zero or got is None or float(got.abs().max()) == 0.0, k
            continue
        assert got is not None, k
        got = got.detach().double().flatten()
        idx = sample_index(got.numel(), GRAD_SAMPLES)
        tol = rtol * amax[i] + atol
        assert (got[idx] - samples[i, :idx.numel()]).abs().max() <= tol, k
        assert abs(got.abs().max() - amax[i]) <= tol, k
        assert abs(got.norm() - norm[i]) <= rtol * norm[i] + atol, k


def check_grads_norm(z, case, grads, rtol, total_frac):
    """As check_grads, for a norm-wise tolerance ||got - want|| <= rtol * ||want|| + total_frac * ||all gradients||: the
    sampled entries and the norm, which that bound also bounds."""
    norm, samples = torch.from_numpy(z[case + '.grad_norm']).double(), torch.from_numpy(z[case + '.grad_samples']).double()
    total = float(z[case + '.grad_total'])
    for i, k in enumerate(z[case + '.names']):
        if torch.isnan(norm[i]):
            continue
        got = grads[str(k)].detach().double().flatten()
        idx = sample_index(got.numel(), GRAD_SAMPLES)
        tol = rtol * norm[i] + total_frac * total
        assert (got[idx] - samples[i, :idx.numel()]).norm() <= tol, k
        assert abs(got.norm() - norm[i]) <= tol, k


def pred_sample(z, case, got):
    """(sample of `got`, stored sample of the reference's tensor) after checking the shapes agree."""
    assert tuple(got.shape) == tuple(z[case + '.pred_shape']), (tuple(got.shape), z[case + '.pred_shape'])
    return got.detach().flatten()[sample_index(got.numel(), PRED_SAMPLES)], torch.from_numpy(z[case + '.pred_samples'])


# ----------------------------------------------------------------------------------------------------------------------
# minting (needs the reference)

class _Writer:
    def __init__(self, ref):
        self.ref, self.out = ref, {}

    def model(self, name, ctor, seed, weight_seed):
        """Build the reference module with `ctor`, replace its weights by the stored recipe, return it."""
        from oracle import e2tts_oracle as O
        torch.manual_seed(seed)
        random.seed(seed)      # the hyper-connections draw their initial stream with python's randrange (SURVEY A.5)
        m = ctor()
        sd = O.randomize_zero_init(m.state_dict(), seed=seed)
        torch.manual_seed(seed + 1)
        random.seed(seed + 1)
        fixed = {k for k, v in ctor().state_dict().items() if torch.equal(v, sd[k])} - set(dict(m.named_parameters()))
        keys = [k for k in sorted(sd) if k not in fixed]   # parameters + buffers drawn at random
        assert all(sd[k].is_floating_point() for k in keys)
        self.out[name + '.names'] = np.array(keys)
        self.out[name + '.shapes'] = np.array([','.join(str(s) for s in sd[k].shape) for k in keys])
        self.out[name + '.is_param'] = np.array([k in dict(m.named_parameters()) for k in keys])
        self.out[name + '.moments'] = np.array([[float(sd[k].mean()), float(sd[k].std()) if sd[k].numel() > 1 else 0.0]
                                                for k in keys], dtype=np.float32)
        small = [sd[k].flatten() for k, (_, std) in zip(keys, self.out[name + '.moments']) if std != 0 and sd[k].numel() <= EXACT_NUMEL]
        self.out[name + '.exact'] = torch.cat(small).numpy() if small else np.zeros(0, dtype=np.float32)
        missing, unexpected = m.load_state_dict(weights(self.out, name, weight_seed), strict=False)
        assert set(missing) == fixed and not unexpected, (missing, unexpected)
        return m

    def grads(self, case, module):
        names, params = self.out[case + '.names'], dict(module.named_parameters())
        amax = np.full(len(names), np.nan, dtype=np.float32)
        norm = np.full(len(names), np.nan, dtype=np.float32)
        samples = np.full((len(names), GRAD_SAMPLES), np.nan, dtype=np.float32)
        flat = []
        for i, k in enumerate(names):
            if k not in params or params[k].grad is None:
                continue
            g = params[k].grad.detach().flatten()
            flat.append(g)
            amax[i], norm[i] = float(g.abs().max()), float(g.norm())
            idx = sample_index(g.numel(), GRAD_SAMPLES)
            samples[i, :idx.numel()] = g[idx].numpy()
        self.out.update({case + '.grad_amax': amax, case + '.grad_norm': norm,
                         case + '.grad_samples': samples, case + '.grad_total': np.float32(torch.cat(flat).norm().item())})

    def pred(self, case, t):
        t = t.detach()
        self.out[case + '.pred_shape'] = np.array(t.shape)
        self.out[case + '.pred_samples'] = t.flatten()[sample_index(t.numel(), PRED_SAMPLES)].numpy()

    def forward_case(self, case, model, mel, text, lens, drop_text_cond, x0_seed):
        from oracle.load_reference import run_reference_forward
        out, rec = run_reference_forward(self.ref, model, mel, text, lens=lens, drop_text_cond=drop_text_cond, x0_seed=x0_seed)
        out.loss.backward()
        assert torch.equal(rec['x0'], randn(mel.shape, x0_seed))
        self.out[case + '.times'] = rec['times'].numpy()
        self.out[case + '.span_mask'] = rec['span_mask'].numpy()
        self.out[case + '.loss'] = np.float32(out.loss.item())
        self.pred(case, out.pred_flow)
        self.grads(case, model)


def e2tts_ctor(ref, transformer=None, **kw):
    return lambda: ref.E2TTS(transformer=dict(dropout=0., max_seq_len=128, **(transformer or KW)), use_vocos=False, **kw)


def main():
    from oracle.load_reference import TorchRecorder, load_reference
    ref = load_reference()
    w = _Writer(ref)

    # forward + backward, every switch the product builds
    fwd = dict(fwd_d2=(2, dict(KW, depth=2), {}, [2, 80], None, ['abc', 'a longer text than the first'], False),
               fwd_d4=(4, dict(KW, depth=4), {}, [2, 80], [80, 51], ['abc', 'a longer text than the first'], False),
               drop=(21, dict(KW, heads=4), {}, [3, 64], [64, 40, 17], ['one', 'two words', ''], True),
               concat=(29, KW, dict(concat_cond=True), [2, 64], [64, 41], ['abc', 'defgh ij'], False),
               interp=(27, KW, dict(interpolated_text=True), [3, 64], [64, 45, 30], ['abc', 'a much longer piece of text', 'xy'], False),
               fourier=(23, dict(KW, attn_fourier_embed_input=True), {}, [2, 64], [64, 45], ['abc', 'defgh ij'], False))
    for case, (seed, tkw, ekw, (b, n), lens, text, drop) in fwd.items():
        model = w.model(case, e2tts_ctor(ref, tkw, **ekw), seed, seed)
        mel = randn((b, n, 100), 100 + seed)
        w.forward_case(case, model, mel, text, torch.tensor(lens) if lens else None, drop, 200 + seed)

    # sample(): one model, three (steps, cfg_strength, duration) cases; y0 drawn from a seeded generator
    model = w.model('sample', e2tts_ctor(ref), 31, 31)
    model.eval()
    for i, (steps, cfg_strength, duration) in enumerate(SAMPLE_CASES):
        rec = TorchRecorder(ref.torch, seed=300 + i)
        ref.torch = rec
        try:
            with torch.no_grad():
                dur = torch.tensor(duration) if isinstance(duration, list) else duration
                out = model.sample(randn((2, 20, 100), 131), text=['Hello', 'Goodbye then'], duration=dur, steps=steps,
                                   cfg_strength=cfg_strength, return_raw_output=True)
        finally:
            ref.torch = rec._t
        y0 = rec.log['randn_like'][0]
        w.out[f'sample{i}.y0_shape'] = np.array(y0.shape)
        w.pred(f'sample{i}', out)

    # DurationPredictor: the prefix fraction is the reference's own draw under torch.manual_seed(5)
    dp = w.model('duration', lambda: ref.DurationPredictor(transformer=dict(dropout=0., max_seq_len=128, **KW)), 41, 41)
    torch.manual_seed(5)
    loss = dp(randn((3, 72, 100), 141), text=['abc', 'hello world', 'x'], lens=torch.tensor([72, 50, 31]))
    loss.backward()
    torch.manual_seed(5)
    w.out['duration.rand_frac'] = torch.zeros(3).uniform_(0, 1).numpy()     # the draw of e2_tts.py:1082 under that seed
    w.out['duration.loss'] = np.float32(loss.item())
    w.grads('duration', dp)

    # velocity-consistency loss with an EMA model
    model = w.model('velocity', e2tts_ctor(ref, velocity_consistency_weight=0.7), 5, 5)
    ema = w.model('velocity_ema', e2tts_ctor(ref), 6, 6)
    ema.eval()
    rec = TorchRecorder(ref.torch, seed=205)
    span = {}
    orig = ref.mask_from_frac_lengths

    def mffl(*a, **k):
        span['mask'] = orig(*a, **k)
        return span['mask'].clone()

    model.cond_drop_prob = -1.0
    lens = torch.tensor([64, 50])
    ref.torch, ref.mask_from_frac_lengths = rec, mffl
    try:
        out = model(randn((2, 64, 100), 105), text=['abc', 'some text'], lens=lens, velocity_consistency_model=ema,
                    velocity_consistency_delta=1e-3)
    finally:
        ref.torch, ref.mask_from_frac_lengths = rec._t, orig
    out.loss.backward()
    w.out.update({'velocity.times': rec.log['rand'][0].numpy(), 'velocity.span_mask': (span['mask'] & ref.lens_to_mask(lens, length=64)).numpy(),
                  'velocity.loss': np.float32(out.loss.item()), 'velocity.flow_loss': np.float32(out.loss_breakdown.flow.item()),
                  'velocity.velocity_loss': np.float32(out.loss_breakdown.velocity_consistency.item())})
    w.grads('velocity', model)

    # parameter names and shapes of the variants
    sd = ref.E2TTS(transformer=dict(dim=128, depth=2, heads=2, attn_fourier_embed_input=True), use_vocos=False, interpolated_text=True,
                   concat_cond=True).state_dict()
    w.out['variants.names'] = np.array(list(sd))
    w.out['variants.shapes'] = np.array([','.join(str(s) for s in v.shape) for v in sd.values()])

    # MelSpec
    w.out['melspec.mel'] = ref.MelSpec()(randn((1, 256 * 10 + 17), 9)).numpy()

    # mask helpers on 200 seeded ragged cases (same torch RNG state -> same rand_like draw), bits packed row-major
    g = torch.Generator().manual_seed(0)
    bits = dict(frac=[], lens_n=[], lens=[])
    for case in range(200):
        b = int(torch.randint(1, 9, (1,), generator=g))
        n = int(torch.randint(8, 300, (1,), generator=g))
        lens = torch.randint(1, n + 1, (b,), generator=g)
        if case % 3 == 0:
            lens[int(torch.randint(0, b, (1,), generator=g))] = n
        frac = torch.rand(b, generator=g) * 0.3 + 0.7          # frac_lengths_mask = (0.7, 1.0), e2_tts.py:1133
        torch.manual_seed(1000 + case)
        bits['frac'].append(ref.mask_from_frac_lengths(lens, frac, max_length=n).flatten())
        bits['lens_n'].append(ref.lens_to_mask(lens, length=n).flatten())
        bits['lens'].append(ref.lens_to_mask(lens).flatten())
    for k, v in bits.items():
        w.out['masks.' + k] = np.packbits(torch.cat(v).numpy())
    w.out['masks.text_ids'] = ref.list_str_to_tensor(['Hello', 'Goodbye', 'héllo wörld']).numpy()

    # an .npz written member by member with a fixed timestamp: minting twice gives the same bytes
    with zipfile.ZipFile(PATH, 'w', compression=zipfile.ZIP_DEFLATED) as f:
        for k in sorted(w.out):
            info = zipfile.ZipInfo(k + '.npy', date_time=(1980, 1, 1, 0, 0, 0))
            info.compress_type = zipfile.ZIP_DEFLATED
            with f.open(info, 'w') as m:
                np.lib.format.write_array(m, np.asarray(w.out[k]), allow_pickle=False)
    print(PATH, os.path.getsize(PATH) // 1024, 'KiB')


if __name__ == '__main__':
    sys.path.insert(0, ROOT)
    main()
