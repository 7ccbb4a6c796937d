"""Load the reference's OWN e2_tts.py, unmodified, by file path (build container only).

TEST INFRASTRUCTURE. The reference tree is not part of this repository, so this module is used only
by the scripts that mint the golden vectors under tests/golden/ (`oracle/make_golden.py`,
`oracle/reference_cases.py`); the tests compare against those vectors.
The reference's seven unvendored third-party imports resolve to `oracle/ref_leaves/` (restated
semantics, SURVEY.md Appendix A) — `e2_tts_pytorch/__init__.py` is bypassed because it pulls in
trainer.py -> matplotlib/accelerate which are not installed.
"""
import importlib.util
import os
import sys

REF_FILE = os.environ.get('E2TTS_REFERENCE_FILE', '/root/reference/e2_tts_pytorch/e2_tts.py')
_LEAVES = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'ref_leaves')
_cached = None


def reference_available():
    return os.path.isfile(REF_FILE)


def load_reference():
    """Returns the reference module object (classes E2TTS, DurationPredictor, Transformer, MelSpec...)."""
    global _cached
    if _cached is not None:
        return _cached
    if not reference_available():
        raise FileNotFoundError(REF_FILE)
    sys.path.insert(0, _LEAVES)
    try:
        spec = importlib.util.spec_from_file_location('_e2tts_reference', REF_FILE)
        mod = importlib.util.module_from_spec(spec)
        sys.modules['_e2tts_reference'] = mod
        spec.loader.exec_module(mod)
    finally:
        sys.path.remove(_LEAVES)
    _cached = mod
    return mod


class TorchRecorder:
    """Proxy for the `torch` global inside the reference module: records the random draws of
    E2TTS.forward (e2_tts.py:1504 uniform_, :201 rand_like, :1519 randn_like, :1523 rand) so the
    same (x0, times, span mask) can be injected into the oracle and the CUDA path. With `seed`, the randn_like
    draws come from a torch.Generator seeded with it, so the first one can be redrawn without the reference."""

    def __init__(self, torch_mod, seed=None):
        self._t = torch_mod
        self.log = {}
        self._gen = None if seed is None else torch_mod.Generator().manual_seed(seed)

    def __getattr__(self, name):
        return getattr(self._t, name)

    def randn_like(self, *a, **k):
        if self._gen is None:
            out = self._t.randn_like(*a, **k)
        else:
            x = a[0]
            out = self._t.randn(x.shape, generator=self._gen, dtype=x.dtype).to(x.device)
        self.log.setdefault('randn_like', []).append(out.clone())
        return out

    def rand(self, *a, **k):
        out = self._t.rand(*a, **k)
        self.log.setdefault('rand', []).append(out.clone())
        return out


def run_reference_forward(ref, model, mel, text, lens=None, drop_text_cond=False, x0_seed=None):
    """Runs reference E2TTS.forward recording x0 / times / span mask. `drop_text_cond` is forced by
    temporarily pinning cond_drop_prob (e2_tts.py:1261 uses python random()). `x0_seed`: see TorchRecorder."""
    rec = TorchRecorder(ref.torch, seed=x0_seed)
    span = {}
    orig_mffl = ref.mask_from_frac_lengths

    def mffl(*a, **k):
        out = orig_mffl(*a, **k)
        span['mask'] = out.clone()
        return out

    saved_prob = model.cond_drop_prob
    model.cond_drop_prob = 2.0 if drop_text_cond else -1.0
    ref.torch, ref.mask_from_frac_lengths = rec, mffl
    try:
        out = model(mel, text=text, lens=lens)
    finally:
        ref.torch, ref.mask_from_frac_lengths = rec._t, orig_mffl
        model.cond_drop_prob = saved_prob
    x0 = rec.log['randn_like'][0]
    times = rec.log['rand'][0]
    span_mask = span['mask']
    if lens is not None:
        span_mask = span_mask & ref.lens_to_mask(lens, length=mel.shape[1])
    return out, dict(x0=x0, times=times, span_mask=span_mask)
