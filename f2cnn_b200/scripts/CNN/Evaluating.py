"""GPU front end behind the names of the reference's scripts/CNN/Evaluating.py.

What the reference does per utterance (EvaluateOneWavArray, reference :27-113): filterbank and
envelope, then 25 s of pure-Python dense framing (:70-78), ~1 s of per-frame normalizeInput
(:79-80), then Keras prediction, an accuracy heuristic and a matplotlib figure.  Here everything
up to the scores is ONE filterbank pass on the GPU: the time-major envelope feeds the
reference network on the tensor cores (api.cnn_evaluate -> csrc/f2_cnn.cu, 3.4 ms for the
46 240 frames of a 3 s utterance) and, transposed, is the matrix the figure shows.  `model` may
be an .npz of the 12 arrays of model.get_weights() (cnn.save_weights) -- no Keras needed -- or
a Keras model, whose weights are then read with get_weights(); a geometry other than the
configured RADIUS = 5 / 128 channels keeps Keras' own predict on the GPU-made frames.  The
accuracy heuristic is counted on the GPU as well (api.label_accuracy; _label_accuracy stays as its
host restatement).  The figure
still belongs to the reference tree (matplotlib) and is imported where the reference needs it.

Public names, signatures, defaults and side effects (files written under OutputWavFiles/,
graphs/) follow the reference; the bodies are organised around small helpers.
"""
import glob
import os
import shutil
import time
from collections import namedtuple
from configparser import ConfigParser

import numpy

from ...gammatone import filters
from ..processing.GammatoneFiltering import GetArrayFromWAV

_Settings = namedtuple("_Settings", "radius dots period_us nchannels lowfreq framerate")


def _settings():
    """configF2CNN.conf of the working directory (the reference re-reads it in every driver)."""
    cfg = ConfigParser()
    cfg.read('configF2CNN.conf')
    radius = cfg.getint('CNN', 'RADIUS')
    return cfg, _Settings(radius, 2 * radius + 1, cfg.getint('CNN', 'SAMPLING_PERIOD'),
                          cfg.getint('FILTERBANK', 'NCHANNELS'), cfg.getint('FILTERBANK', 'LOW_FREQ'),
                          cfg.getint('FILTERBANK', 'FRAMERATE'))


def _bank(framerate, st, centre, coefs):
    """Filterbank of the call, designed on demand like reference :42-49."""
    if centre is None:
        centre = filters.centre_freqs(framerate, st.nchannels, st.lowfreq)
        coefs = filters.make_erb_filters(framerate, centre)
    return centre, coefs


def SNRdbToSNRlinear(SNRdb):
    """dB -> ratio, reference :180-181.  It is a power ratio that the caller applies to an
    amplitude; kept as is."""
    return 10 ** (SNRdb / 10.0)


def RMS(signal):
    """Root mean square, reference :184-190.  numpy.square keeps the dtype of an int16 WAV array,
    so the squares wrap around exactly as they do in the reference (SURVEY.md 8a row 14)."""
    return numpy.sqrt(numpy.mean(numpy.square(signal)))


def MixNoise(wavList, SNRdB):
    """White Gaussian noise of standard deviation RMS(wav) / SNRdbToSNRlinear(SNRdB) added to the
    waveform: float64 output (reference :199-200)."""
    sigma = RMS(wavList) / SNRdbToSNRlinear(SNRdB)
    return numpy.random.normal(scale=sigma, size=wavList.shape[0]) + wavList


def PrepareInputFromArray(wavArray, framerate, config, LPF=False, CUTOFF=100, CENTER_FREQUENCIES=None,
                          FILTERBANK_COEFFICIENTS=None):
    """Everything between the waveform and model.predict: (nb, 2R+1, C) float64 frames, each
    log-min-max normalised, nb = n - (2R+1)*STEP (reference :52-80).  Also returns the bank."""
    from ... import api
    radius = config.getint('CNN', 'RADIUS')
    step = int(framerate * config.getint('CNN', 'SAMPLING_PERIOD') * 1e-6)
    st = _Settings(radius, 2 * radius + 1, 0, config.getint('FILTERBANK', 'NCHANNELS'),
                   config.getint('FILTERBANK', 'LOW_FREQ'), framerate)
    centre, coefs = _bank(framerate, st, CENTER_FREQUENCIES, FILTERBANK_COEFFICIENTS)
    print("Applying filterbank...")
    print("Extraction Envelope with {}Hz Low Pass Filter...".format(CUTOFF) if LPF else "Extracting Envelope...")
    print("Generating input data for CNN...")
    frames = api.dense_frames(wavArray, coefs, LPF, CUTOFF, radius, step, normalize=True, dtype=numpy.float64)
    print("INPUT SHAPE:", frames.shape)
    return frames, centre, coefs, step


def _decisions(scores):
    """1 = rising when the second score wins (reference :87)."""
    return [1 if s[1] > s[0] else 0 for s in scores]


def _label_accuracy(labels, decisions, step):
    """The reference's heuristic (:92-110): a frame index strictly between two consecutive label
    timepoints and closer than STEP to one of them is scored against the nearer label (ties go
    to the earlier one).  Raises ZeroDivisionError when no frame qualifies, like the reference."""
    times = [l[0] for l in labels]
    classes = [l[1] for l in labels]
    hits = 0
    counted = 0
    for frame, decided in enumerate(decisions):
        for left in range(len(labels) - 1):
            lo, hi = times[left], times[left + 1]
            if not (lo < frame < hi):
                continue
            d_lo, d_hi = abs(frame - lo), abs(frame - hi)
            if d_lo >= step and d_hi >= step:
                continue
            target = classes[left] if d_lo <= d_hi else classes[left + 1]
            hits += 1 if decided == target else 0
            counted += 1
    return hits / counted


def _resolve_model(model, st):
    """(weights, keras network): the 12 parameter arrays for the tensor-core kernels when the geometry is
    the configured one, else the Keras network whose predict takes the frames (reference :84-86)."""
    from ... import cnn
    tensor_core = st.dots == 11 and st.nchannels == 128
    for cand in (model, str(model) + '.npz'):
        if str(cand).endswith('.npz') and os.path.isfile(cand):
            if not tensor_core:
                raise ValueError("an .npz model needs the configured geometry (RADIUS = 5, 128 channels)")
            return cnn.load_weights(cand), None
    import keras  # absent here: the reference's own ImportError
    network = keras.models.load_model(model)
    if tensor_core and hasattr(network, 'get_weights'):
        return network.get_weights(), network
    return None, network


def EvaluateOneWavArray(wavArray, framerate, wavFileName, model='last_trained_model', LPF=False, CUTOFF=100,
                        CENTER_FREQUENCIES=None, FILTERBANK_COEFFICIENTS=None):
    """One waveform through front end, CNN and figure (reference :27-113)."""
    from ... import api
    from ..processing.LabelDataGenerator import ExtractLabel
    from ..processing.FBFileReader import ExtractFBFile
    from ..processing.PHNFileReader import ExtractPhonemes
    # the figure is the reference tree's (matplotlib): resolved at call time
    from scripts.plotting.PlottingCNN import PlotEnvelopesAndCNNResultsWithPhonemes

    cfg, st = _settings()
    found = ExtractLabel(wavFileName, cfg)
    labels = None if found is None else [(row[-4], row[-1]) for row in found]

    step = int(framerate * cfg.getint('CNN', 'SAMPLING_PERIOD') * 1e-6)
    centre, coefs = _bank(framerate, st, CENTER_FREQUENCIES, FILTERBANK_COEFFICIENTS)
    print("Applying filterbank...")
    print("Extraction Envelope with {}Hz Low Pass Filter...".format(CUTOFF) if LPF else "Extracting Envelope...")

    stem = os.path.splitext(wavFileName)[0]
    print("Extracting Formants...")
    formants, _ = ExtractFBFile(stem + '.FB')
    print("Extracting Phonemes...")
    phonemes = ExtractPhonemes(stem + '.PHN')

    print("Generating input data for CNN...")
    weights, network = _resolve_model(model, st)
    print("Evaluating the data with the pretrained model...")
    if weights is not None:
        # waveform -> scores on the device; the envelopes come out of the same pass
        scores, envelopes = api.cnn_evaluate(wavArray, coefs, weights, LPF, CUTOFF, st.radius, step)
        print("INPUT SHAPE:", (scores.shape[0], st.dots, st.nchannels))
    else:
        envelopes, frames = api.evaluate_front_end(wavArray, coefs, LPF, CUTOFF, st.radius, step)
        print("INPUT SHAPE:", frames.shape)
        scores = network.predict(frames.reshape(frames.shape[0], st.dots, st.nchannels, 1), verbose=1)
        del frames
    if network is not None:
        import keras
        keras.backend.clear_session()
        del network

    accuracy = None
    if labels is not None:
        # the reference's heuristic (:87-110) on the GPU; hits / counted raises ZeroDivisionError as it does there
        hits, counted = api.label_accuracy(scores, labels, step)
        accuracy = hits / counted
    print("Plotting...")
    PlotEnvelopesAndCNNResultsWithPhonemes(envelopes, scores, accuracy, centre, phonemes, formants, wavFileName)


def EvaluateOneWavFile(file, LPF=False, CUTOFF=50, model='last_trained_model', CENTER_FREQUENCIES=None,
                       FILTERBANK_COEFFICIENTS=None):
    """Read one .WAV (RIFF or NIST SPHERE) and evaluate it (reference :116-137)."""
    print('Using model', model)
    print("File:\t\t{}".format(file))
    rate, samples = GetArrayFromWAV(file)
    EvaluateOneWavArray(samples, rate, file, model=model, LPF=LPF, CUTOFF=CUTOFF,
                        CENTER_FREQUENCIES=CENTER_FREQUENCIES, FILTERBANK_COEFFICIENTS=FILTERBANK_COEFFICIENTS)
    print("\t\t{}\tdone !".format(file))


def EvaluateRandom(count=None, LPF=False, CUTOFF=50):
    """Evaluate the organised .WAV files in random order, all of them or `count` draws with
    replacement (reference :140-177)."""
    os.environ['TF_CPP_MIN_LOG_LEVEL'] = '3'
    started = time.time()
    if not os.path.isdir("graphs"):
        os.makedirs(os.path.join('graphs', 'FallingOrRising'))
    candidates = glob.glob(os.path.join('resources', 'f2cnn', '*', '*.WAV'))
    # like the reference, the banner indexes the list before the emptiness check
    print("\n###############################\nEvaluating network on {} WAV files in '{}'.".format(
        len(candidates), os.path.split(candidates[0])[0]))
    if not candidates:
        print("NO WAV FILES FOUND")
        exit(-1)
    _, st = _settings()
    centre, coefs = _bank(st.framerate, st, None, None)
    if count is None:
        numpy.random.shuffle(candidates)
    elif count > 1:
        candidates = numpy.random.choice(candidates, count)
    for path in candidates:
        EvaluateOneWavFile(path, LPF=LPF, CUTOFF=CUTOFF, CENTER_FREQUENCIES=centre, FILTERBANK_COEFFICIENTS=coefs)
    print("Evaluating network on all files.")
    print('              Total time:', time.time() - started)
    print('')


def _copy_sidecars(src_stem, dst_stem):
    """.FB / .PHN / .WRD next to the noisy copy, if the originals exist (reference :210-216)."""
    try:
        for ext in ('.FB', '.PHN', '.WRD'):
            shutil.copyfile(src_stem + ext, dst_stem + ext)
    except FileNotFoundError as err:
        print(err.strerror)
        print("No .FB or .PHN or .WRD files.")


def EvaluateWithNoise(file, LPF=False, CUTOFF=100, model='last_trained_model', CENTER_FREQUENCIES=None,
                      FILTERBANK_COEFFICIENTS=None, SNRdB=-3):
    """Add noise at SNRdB, save OutputWavFiles/addedNoise/<name><SNR>dB.WAV (float64 samples, as
    the reference writes them) with its sidecar files, then evaluate it (reference :193-221)."""
    from scipy.io import wavfile
    print("File:\t\t{}".format(file))
    print("Appyling gaussian noise, new SNR is {SNR}dB".format(SNR=SNRdB))
    rate, clean = GetArrayFromWAV(file)
    noisy = MixNoise(clean, SNRdB)

    out_dir = os.path.join('OutputWavFiles', 'addedNoise')
    os.makedirs(out_dir, exist_ok=True)
    src_stem = os.path.splitext(file)[0]
    dst_stem = os.path.join(out_dir, os.path.basename(src_stem)) + '{SNR}dB'.format(SNR=SNRdB)
    noisy_path = dst_stem + '.WAV'
    wavfile.write(noisy_path, rate, noisy)
    _copy_sidecars(src_stem, dst_stem)
    print('New noisy WAVE file saved as', noisy_path)

    EvaluateOneWavArray(noisy, rate, noisy_path, model=model, LPF=LPF, CUTOFF=CUTOFF,
                        CENTER_FREQUENCIES=CENTER_FREQUENCIES, FILTERBANK_COEFFICIENTS=FILTERBANK_COEFFICIENTS)
    print("\t\t{}\tdone !".format(file))
