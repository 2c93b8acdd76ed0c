"""The reference's OWN entry points on the drop-in (needs a checkout of the original F2CNN tree named by
F2CNN_REFERENCE; skipped without one): after dropin.install() the reference's unmodified f2cnn.py imports,
every dispatch name it binds (f2cnn.py:4-9, 27-45) resolves to this package, a late install()
re-binds the names PlottingProcessing.py:12-15 imported by value, and every public function of the
shadowed modules has the reference's signature."""
import importlib
import inspect
import os
import sys
import types

import pytest

REF = os.environ.get("F2CNN_REFERENCE", "")
pytestmark = pytest.mark.skipif(not (REF and os.path.isfile(os.path.join(REF, "f2cnn.py"))),
                                reason="F2CNN_REFERENCE does not name a reference tree")

SHADOWED = ["gammatone.filters", "scripts.processing.GammatoneFiltering", "scripts.processing.EnvelopeExtraction",
            "scripts.processing.InputGenerator", "scripts.processing.LabelDataGenerator",
            "scripts.processing.FBFileReader", "scripts.processing.PHNFileReader", "scripts.CNN.Evaluating"]


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


@pytest.fixture
def clean_modules():
    """Import state of this process is restored afterwards: the reference must not leak into other tests."""
    saved_modules = dict(sys.modules)
    saved_path = list(sys.path)
    # third-party modules the reference imports at module level and this image lacks; never called here
    if "sphfile" not in sys.modules:
        _stub("sphfile", SPHFile=object)
    try:
        importlib.import_module("matplotlib")
    except ImportError:
        mpl = _stub("matplotlib")
        mpl.pyplot = _stub("matplotlib.pyplot")
        mpl.colors = _stub("matplotlib.colors", LogNorm=object)
    for name in list(sys.modules):
        if name == "f2cnn" or name == "configure" or name.split(".")[0] in ("scripts", "gammatone"):
            del sys.modules[name]
    sys.path.insert(0, REF)
    yield
    from f2cnn_b200 import dropin
    dropin.uninstall()
    sys.path[:] = saved_path
    for name in list(sys.modules):
        if name not in saved_modules:
            del sys.modules[name]
    sys.modules.update(saved_modules)


def _public_functions(mod):
    return {n: f for n, f in vars(mod).items()
            if inspect.isfunction(f) and not n.startswith("_") and f.__module__ == mod.__name__}


def test_reference_cli_binds_to_the_dropin_and_signatures_match(clean_modules):
    # 1. the reference as it is: signatures of every public function of the modules we shadow
    ref_sigs = {}
    for name in SHADOWED:
        mod = importlib.import_module(name)
        assert mod.__file__.startswith(REF), name
        ref_sigs[name] = {n: inspect.signature(f) for n, f in _public_functions(mod).items()}
    for name in list(sys.modules):
        if name.split(".")[0] in ("scripts", "gammatone"):
            del sys.modules[name]
    # 2. drop-in first, then the reference's own CLI module
    from f2cnn_b200 import dropin
    installed = dropin.install()
    f2cnn = importlib.import_module("f2cnn")
    assert f2cnn.__file__ == os.path.join(REF, "f2cnn.py")
    for attr in ("FilterAllOrganisedFiles", "ExtractAllEnvelopes", "GenerateInputData", "GenerateLabelData",
                 "EvaluateOneWavFile", "EvaluateRandom", "EvaluateWithNoise"):
        assert getattr(f2cnn, attr).__module__.startswith("f2cnn_b200."), attr
    # what the drop-in does not replace keeps coming from the reference tree
    assert f2cnn.OrganiseAllFiles.__module__ == "scripts.processing.OrganiseFiles"
    assert sys.modules["scripts.processing.OrganiseFiles"].__file__.startswith(REF)
    assert f2cnn.PlotEnvelopesAndFormantsFromFile.__module__ == "f2cnn_b200.scripts.plotting.PlottingProcessing"
    # 3. every public function of the reference exists here with the same signature
    diffs = []
    for name in SHADOWED:
        ours = _public_functions(installed[name])
        for fn, sig in ref_sigs[name].items():
            if fn not in ours:
                diffs.append("%s.%s missing" % (name, fn))
            elif inspect.signature(ours[fn]) != sig:
                diffs.append("%s.%s%s != reference %s" % (name, fn, inspect.signature(ours[fn]), sig))
    assert not diffs, "\n".join(diffs)
    for const in ("DEFAULT_FILTER_NUM", "DEFAULT_LOW_FREQ", "DEFAULT_HIGH_FREQ"):
        assert hasattr(installed["gammatone.filters"], const)


def test_late_install_rebinds_names_imported_by_value(clean_modules):
    """PlottingProcessing.py:12-15 and f2cnn.py:4-9 use `from ... import name`: a reference that was
    imported BEFORE install() must not stay on the CPU filterbank."""
    plotting = importlib.import_module("scripts.plotting.PlottingProcessing")
    f2cnn = importlib.import_module("f2cnn")
    assert plotting.GetFilteredOutputFromFile.__module__ == "scripts.processing.GammatoneFiltering"
    assert plotting.GetFilteredOutputFromFile.__code__.co_filename.startswith(REF)
    from f2cnn_b200 import dropin
    dropin.install()
    for attr in ("centre_freqs", "make_erb_filters", "ExtractEnvelopeFromMatrix", "ExtractFBFile",
                 "GetFilteredOutputFromFile", "GetArrayFromWAV"):
        fn = getattr(plotting, attr)
        assert fn.__module__.startswith("f2cnn_b200."), attr
    for attr in ("FilterAllOrganisedFiles", "ExtractAllEnvelopes", "GenerateInputData", "GenerateLabelData",
                 "EvaluateOneWavFile", "EvaluateRandom", "EvaluateWithNoise", "PlotEnvelopesAndFormantsFromFile"):
        assert getattr(f2cnn, attr).__module__.startswith("f2cnn_b200."), attr
    # every name the reference module imports from a shadowed module is covered by the re-bind table
    import ast
    src = open(os.path.join(REF, "scripts", "plotting", "PlottingProcessing.py")).read()
    imported = {a.name for node in ast.walk(ast.parse(src)) if isinstance(node, ast.ImportFrom)
                and node.module in dropin._MODULES for a in node.names}
    assert imported == set(dropin._REBIND["scripts.plotting.PlottingProcessing"])


def test_gammatonegram_reshape_equals_the_reference(clean_modules):
    """scripts/plotting/PlottingProcessing.py:18-60 (ERB row heights, row repetition, column slice) against the
    drop-in's, and the signatures of its public functions (`axis` aside: the reference binds pyplot there)."""
    import numpy as np
    ref = importlib.import_module("scripts.plotting.PlottingProcessing")
    assert ref.__file__.startswith(REF)
    ours = importlib.import_module("f2cnn_b200.scripts.plotting.PlottingProcessing")
    from f2cnn_b200.gammatone import filters
    rng = np.random.default_rng(3)
    for C, low in ((128, 100), (37, 50), (256, 20)):
        cfs = filters.centre_freqs(16000, C, low)
        env = rng.random((C, 300))
        assert ours.GetNewHeightERB(env, cfs) == ref.GetNewHeightERB(env, cfs)
        for start, end in ((0, None), (17, None), (5, 120)):
            assert np.array_equal(ours.ReshapeEnvelopesForSpectrogram(env, cfs, start, end),
                                  ref.ReshapeEnvelopesForSpectrogram(env, cfs, start, end))
    for name, fn in _public_functions(ref).items():
        theirs = [(p.name, p.default) for p in inspect.signature(fn).parameters.values() if p.name != "axis"]
        mine = [(p.name, p.default) for p in inspect.signature(getattr(ours, name)).parameters.values()
                if p.name not in ("axis", "NYQUIST")]
        assert mine == theirs, name
