"""GPU implementation behind the names of the reference's scripts/processing/InputGenerator.py.

Contract kept from the reference (file:line there):
  * GetListOfEnvelopeFilesAndTimepoints (:9-25): label CSV -> {"<TEST|TRAIN>/<DRr>.<SPKR>.<SENT>.
    ENV1.npy": [timepoints, in CSV order]}.
  * GenerateInputData (:28-93): rows ordered by SORTED file key, CSV order inside a file (:50,
    :67-82); row = the envelope samples at center + STEP*(j - RADIUS), j = 0..2*RADIUS (:76);
    float64 -> float32 only at the end (:83); saved as trainingData/input_data_LPF<k>.npy,
    input_data_NOLPF.npy or `inputFile`, plus trainingData/last_input_data.npy (:86-90);
    `print` + exit(-1) when there is nothing to do (:32-34, :46-48).
The window gather runs on the GPU (float64 -> float32 on the device rounds to nearest even like
numpy.astype).  Extension: an utterance whose .ENV1.npy is missing but whose .WAV is present is
computed by the fused filterbank+envelope kernel, all such utterances in ONE batched launch
sequence (the reference would stop with FileNotFoundError).
Extension: GenerateInputDataSweep writes the input_data_LPF<k>.npy / input_data_NOLPF.npy of
several cutoffs from one filterbank pass over the .WAV files.
"""
import csv
import os
import time
from collections import OrderedDict
from configparser import ConfigParser

import numpy

_ROOT = os.path.join('resources', 'f2cnn')
_OUT_DIR = 'trainingData'


def GetListOfEnvelopeFilesAndTimepoints(labelFilename):
    table = OrderedDict()
    with open(labelFilename, 'r') as handle:
        for record in csv.reader(handle):
            split, region, speaker, sentence, _phoneme, timepoint = record[:6]
            if len(record) != 9:
                raise ValueError("not enough values to unpack (expected 9, got {})".format(len(record)))
            name = '.'.join((region, speaker, sentence, 'ENV1.npy'))
            table.setdefault(os.path.join(split, name), []).append(int(timepoint))
    return dict(table)


def _geometry():
    cfg = ConfigParser()
    cfg.read('configF2CNN.conf')
    radius = cfg.getint('CNN', 'RADIUS')
    rate = cfg.getint('FILTERBANK', 'FRAMERATE')
    step = int(rate * cfg.getint('CNN', 'SAMPLING_PERIOD') / 1000000)
    return cfg, radius, step, rate, cfg.getint('FILTERBANK', 'NCHANNELS')


def _say_lpf(LPF, CUTOFF):
    print("Using Low Pass Filtering with a cutoff at {}Hz".format(CUTOFF) if LPF else "Not using Low Pass Filtering")


def _bank_and_waves(paths, cfg, rate, channels):
    """The configured filterbank and the waveforms of `paths` (features_to_windows' `waves` argument)."""
    from concurrent.futures import ThreadPoolExecutor
    from ... import ingest
    from ...gammatone import filters
    from .GammatoneFiltering import GetArrayFromWAV
    low = cfg.getint('FILTERBANK', 'LOW_FREQ')
    coefs = filters.make_erb_filters(rate, filters.centre_freqs(rate, channels, low))
    try:  # mono 16-bit PCM (TIMIT): straight into one pinned buffer
        flat, lengths, _ = ingest.read_corpus(paths)
        return coefs, (flat, lengths)
    except ValueError:  # anything else (e.g. the float64 WAVs of `cnn evalnoise`): decode file by file
        with ThreadPoolExecutor(max_workers=8) as readers:
            return coefs, [samples for _, samples in readers.map(GetArrayFromWAV, paths)]


def _fill_from_waveforms(pending, out, cfg, rate, channels, radius, step, LPF, CUTOFF):
    """pending: [(first row, wav path, timepoints)].  One batch for all of them."""
    from ... import api
    coefs, waves = _bank_and_waves([p[1] for p in pending], cfg, rate, channels)
    rows = api.features_to_windows(waves, coefs, [p[2] for p in pending], LPF, CUTOFF, radius, step)
    cursor = 0
    for first, _, points in pending:
        out[first:first + len(points)] = rows[cursor:cursor + len(points)]
        cursor += len(points)


def GenerateInputData(labelFile=None, inputFile=None, LPF=False, CUTOFF=100):
    from ... import api
    started = time.time()
    if not os.path.isdir(_OUT_DIR):
        print("LABEL GENERATION SHOULD BE DONE PRIOR TO INPUT...")
        exit(-1)
    labels = labelFile or os.path.join(_OUT_DIR, "label_data.csv")
    per_file = GetListOfEnvelopeFilesAndTimepoints(labels)
    print("\n###############################\nGenerating Input Data from files with '{}'.".format(labels))
    _say_lpf(LPF, CUTOFF)
    if not per_file:
        print("NO ENV1.npy FILES FOUND, PLEASE GENERATE ENVELOPES")
        exit(-1)
    order = sorted(per_file)
    total = sum(len(v) for v in per_file.values())
    print(len(order), "files found along with their", total, "entry timepoints.")

    cfg, radius, step, rate, channels = _geometry()
    data = numpy.zeros((total, 2 * radius + 1, channels), dtype=numpy.float32)
    print("Output shape:", data.shape)

    row = 0
    pending = []
    for done, key in enumerate(order, start=1):
        points = per_file[key]
        saved = os.path.join(_ROOT, key)
        print("Reading:\t{}".format(saved))
        if os.path.isfile(saved):
            envelope = numpy.load(saved)
            if envelope.shape[0] != channels:
                raise ValueError("could not broadcast input array from shape ({},) into shape ({},)".format(
                    envelope.shape[0], channels))
            data[row:row + len(points)] = api.gather_windows_from_matrix(envelope, points, radius, step)
        else:
            wave_path = saved[:-len('.ENV1.npy')] + '.WAV'
            if not os.path.isfile(wave_path):
                raise FileNotFoundError(2, 'No such file or directory', saved)
            pending.append((row, wave_path, points))
        row += len(points)
        print("\t\t{:<50} done !  {}/{} Files".format(saved, done, len(order)))
    if pending:
        _fill_from_waveforms(pending, data, cfg, rate, channels, radius, step, LPF, CUTOFF)
    print('Generated Input Matrix of shape {}.'.format(data.shape))

    default_name = 'input_data_LPF{}.npy'.format(CUTOFF) if LPF else 'input_data_NOLPF.npy'
    target = inputFile or os.path.join(_OUT_DIR, default_name)
    print("Saving as {}...".format(target))
    os.makedirs(os.path.split(target)[0], exist_ok=True)
    numpy.save(target, data)
    numpy.save(os.path.join(_OUT_DIR, 'last_input_data.npy'), data)  # the reference's "just in case" copy
    print('                Total time:', time.time() - started)
    print('')


def GenerateInputDataSweep(labelFile=None, CUTOFFS=(20, 50, 100)):
    """GenerateInputData for several cutoffs at once: trainingData/input_data_LPF<k>.npy for every k of
    CUTOFFS, input_data_NOLPF.npy for an entry None, rows ordered as GenerateInputData orders them.  The
    filterbank and the Hilbert transform run once for all cutoffs (api.features_to_windows_sweep), so the
    envelopes always come from the .WAV files: an .ENV1.npy on disk holds one cutoff and cannot serve a
    sweep.  A missing .WAV raises FileNotFoundError.  Unlike GenerateInputData, no
    trainingData/last_input_data.npy is written: there is no single last input."""
    from ... import api
    started = time.time()
    if not os.path.isdir(_OUT_DIR):
        print("LABEL GENERATION SHOULD BE DONE PRIOR TO INPUT...")
        exit(-1)
    cutoffs = list(CUTOFFS)
    labels = labelFile or os.path.join(_OUT_DIR, "label_data.csv")
    per_file = GetListOfEnvelopeFilesAndTimepoints(labels)
    print("\n###############################\nGenerating Input Data from files with '{}'.".format(labels))
    for cutoff in cutoffs:
        _say_lpf(cutoff is not None, cutoff)
    if not per_file:
        print("NO ENV1.npy FILES FOUND, PLEASE GENERATE ENVELOPES")
        exit(-1)
    order = sorted(per_file)
    total = sum(len(v) for v in per_file.values())
    print(len(order), "files found along with their", total, "entry timepoints.")

    cfg, radius, step, rate, channels = _geometry()
    print("Output shape:", (total, 2 * radius + 1, channels), "x", len(cutoffs))
    pending = []
    for done, key in enumerate(order, start=1):
        saved = os.path.join(_ROOT, key)
        wave_path = saved[:-len('.ENV1.npy')] + '.WAV'
        print("Reading:\t{}".format(wave_path))
        if not os.path.isfile(wave_path):
            raise FileNotFoundError(2, 'No such file or directory', wave_path)
        pending.append((wave_path, per_file[key]))
        print("\t\t{:<50} done !  {}/{} Files".format(wave_path, done, len(order)))
    coefs, waves = _bank_and_waves([p[0] for p in pending], cfg, rate, channels)
    planes = api.features_to_windows_sweep(waves, coefs, [p[1] for p in pending], cutoffs, radius, step)

    os.makedirs(_OUT_DIR, exist_ok=True)
    for cutoff, data in zip(cutoffs, planes):
        print('Generated Input Matrix of shape {}.'.format(data.shape))
        name = 'input_data_LPF{}.npy'.format(cutoff) if cutoff is not None else 'input_data_NOLPF.npy'
        target = os.path.join(_OUT_DIR, name)
        print("Saving as {}...".format(target))
        numpy.save(target, data)
    print('                Total time:', time.time() - started)
    print('')

