"""Import shim for the UNMODIFIED reference (never for the product path).

The reference is a checkout of AaronZ345/StyleSinger named by the STYLESINGER_REF environment variable; nothing in the
package or the tests needs it.  Users: tools/make_golden.py (the fixtures under tests/golden/) and baseline/ref_harness.py
(the reference arms of bench.py and tools/baseline_arms.py).  Shims follow SURVEY.md
§8(c): they only satisfy import-time dependencies that are unused on the hot path (librosa, matplotlib, resemblyzer,
parselmouth, skimage, webrtcvad, ... are imported by reference files but never called between `ph` tokens and the
waveform); no hot-path arithmetic is touched.
"""
import importlib.abc
import importlib.machinery
import os
import sys
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def find_reference():
    c = os.environ.get("STYLESINGER_REF")
    return c if c and os.path.isdir(os.path.join(c, "modules", "StyleSinger")) else None


REF = find_reference()


class _Dummy:
    """Stands in for any attribute of a stubbed third-party module (classes, functions, constants)."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Dummy()

    def __getattr__(self, n):
        if n.startswith("__"):
            raise AttributeError(n)
        return _Dummy()


# third-party packages the reference imports at module level but never uses on the ph -> mel -> wav path
_STUBBED = ("librosa", "pycwt", "chardet", "pyloudnorm", "matplotlib", "resemblyzer", "parselmouth", "skimage",
            "webrtcvad", "tensorboardX", "g2p_en", "pypinyin", "jieba", "textgrid", "praatio", "pyworld", "soundfile",
            "torchaudio", "nltk", "inflect", "unidecode", "pretty_midi", "miditoolkit", "h5py", "numba", "sklearn",
            "Levenshtein", "editdistance", "textdistance")


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, name, path=None, target=None):
        # last finder on sys.meta_path: only consulted for names no real finder could resolve
        if name.split(".")[0] in _STUBBED:
            return importlib.machinery.ModuleSpec(name, self, is_package=True)
        return None

    def create_module(self, spec):
        m = types.ModuleType(spec.name)
        m.__path__ = []
        m.__getattr__ = lambda attr: (_ for _ in ()).throw(AttributeError(attr)) if attr.startswith("__") else _Dummy
        return m

    def exec_module(self, module):
        if module.__name__ == "matplotlib":
            module.use = lambda *a, **k: None


_finder = None


def install(T=100, f0_T=None, overrides=None):
    """chdir to the reference, stub unused imports, load hparams. Returns the reference's global hparams dict."""
    global _finder
    ref = find_reference()
    if ref is None:
        raise RuntimeError("reference not found: set STYLESINGER_REF to a checkout of AaronZ345/StyleSinger")
    if ref not in sys.path:
        sys.path.insert(0, ref)
    os.chdir(ref)
    if _finder is None:
        _finder = _StubFinder()
        sys.meta_path.append(_finder)  # after the real finders: only names nothing else can import are stubbed
    import scipy.signal
    import scipy.signal.windows
    if not hasattr(scipy.signal, "kaiser"):
        scipy.signal.kaiser = scipy.signal.windows.kaiser
    from utils.hparams import set_hparams, hparams
    saved = sys.argv
    sys.argv = [saved[0]]
    try:
        set_hparams(config="egs/stylesinger.yaml", exp_name="", print_hparams=False)
    finally:
        sys.argv = saved
    hparams["timesteps"] = hparams["K_step"] = T
    hparams["f0_timesteps"] = f0_T if f0_T is not None else T
    if overrides:
        hparams.update(overrides)
    return hparams
