"""The f0 track of a soundgen() call, for the device's f0 labels (K12) to be checked against.

The track of a voiced syllable is rebuilt from the artefacts the oracle's generateHarmonics returns (the epochs,
gc_upsampled, pitch_per_gc and the crossings (zc1, zc2) crossFade chose): position q of the joined waveform holds
sample k of epoch e, and its f0 is pitch_upsampled at that sample.  soundgen_f0 is the oracle's soundgen() with the
track carried alongside the samples; its samples equal the oracle's bit for bit (tests/test_f0_host.py), which ties
the layout the track follows to the oracle's.
"""
import math

import numpy as np

from oracle import soundgen_oracle as so
from oracle.rprims import r_round, r_sum
from oracle.soundgen_call import DEFAULT_FORMANTS, _df, rnorm_bounded, wiggleAnchors


def syllable_epoch_map(art, samplingRate):
    """(epoch, k) of every position of the joined waveform of one generateHarmonics call, replaying crossFade
    (R/utilities_soundgen.R:328-375) from its recorded crossings: ampl1 is cut after its zc1-th sample (that sample
    keeps its place in the outgoing epoch, the zero written after it too), ampl2 from its (zc2 + 1)-th, and inside a
    cross-fade of crossLenPoints >= 2 samples the position belongs to the incoming epoch.  The two samples of
    `waveform = 0` and of the zero after it take the first kept sample of epoch 0."""
    gu = art.gc_upsampled
    cross_max = math.floor(15 * samplingRate / 1000)
    ep, kk = np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    for e, (zc1, zc2) in enumerate(art.zc):
        n_e = int(gu[art.epochs[e, 1]] - gu[art.epochs[e, 0] - 1] + 1)
        z2 = zc2 or 0
        k2 = np.arange(z2, n_e, dtype=np.int64)
        if e == 0:        # findZeroCrossing(0, 1) = 1: ampl1 = c(0, 0)
            ep, kk = np.zeros(2, dtype=np.int64), np.full(2, z2, dtype=np.int64)
        elif zc1 is not None:
            ep, kk = ep[:zc1 + 1], kk[:zc1 + 1]
        cl = min(cross_max, ep.size - 1, k2.size - 1)
        keep = ep.size if cl < 2 else ep.size - cl
        ep = np.concatenate((ep[:keep], np.full(k2.size, e, dtype=np.int64)))
        kk = np.concatenate((kk[:keep], k2))
    return ep, kk


def syllable_track(art, samplingRate):
    """f0 of every sample of one generateHarmonics output: pitch_upsampled (utilities_soundgen.R:392-416, from the
    artefacts' pitch_per_gc) at gc_upsampled[start of the sample's epoch] - 1 + k."""
    pu, _ = so.upsample(art.pitch_per_gc, samplingRate)
    ep, kk = syllable_epoch_map(art, samplingRate)
    start = art.gc_upsampled[art.epochs[:, 0] - 1]
    return pu[start[ep] - 1 + kk]


def soundgen_f0(repeatBout=1, nSyl=1, sylLen=300, pauseLen=200,
             pitchAnchors=((0, .1, .9, 1), (100, 150, 135, 100)), pitchAnchorsGlobal=None,
             temperature=0.025, maleFemale=0, creakyBreathy=0, nonlinBalance=0, nonlinDep=50,
             jitterLen=1, jitterDep=3, vibratoFreq=5, vibratoDep=0, shimmerDep=0, attackLen=50,
             rolloff=-12, rolloffOct=-12, rolloffKHz=-6, rolloffParab=0, rolloffParabHarm=3,
             rolloffLip=6, formants='default', formantDep=1, formantDepStoch=30,
             vocalTract=15.5, subFreq=100, subDep=100, shortestEpoch=300, amDep=0, amFreq=30,
             amShape=0, noiseAnchors=((0, 300), (-120, -120)), formantsNoise=None,
             rolloffNoise=-14, mouthAnchors=((0, 1), (.5, .5)), amplAnchors=None,
             amplAnchorsGlobal=None, samplingRate=16000, windowLength=50, overlap=75,
             addSilence=100, pitchFloor=50, pitchCeiling=3500, pitchSamplingRate=3500,
             throwaway=-120, invalidArgAction='adjust', rng=None, contour_method='loess'):
    """oracle.soundgen_call.soundgen (R/soundgen.R:208-862) with the f0 track built alongside the samples: returns
    (sound, f0).  Every statement that draws or shapes the sound is the oracle's, in its order; the f0 lines
    (`*_f0`) follow each concatenation, pad, insertion and length change with the same arguments.  A voiced syllable's
    track is syllable_track(); pauses, silences, noise and zero syllables are 0; the filtered bout keeps the positions
    of `sound` (seewave's istft overlap-adds at the stft frame starts), cut or padded with 0 to its length."""
    rng = rng or so.RStream()
    loc = dict(locals())
    warnings = []
    for p in so.CHECKED_PARS:  # :279-302
        v = loc[p]
        _, lo, hi, _ = so.PERMITTED[p]
        if not isinstance(v, (int, float)) or v < lo or v > hi:
            if invalidArgAction == 'abort':
                raise ValueError('%s must be between %s and %s' % (p, lo, hi))
            elif invalidArgAction == 'ignore':
                warnings.append("%s outside its range in 'permittedValues'" % p)
            else:
                loc[p] = so.PERMITTED[p][0]
                warnings.append('%s outside permitted range, reset to %s' % (p, loc[p]))
    (repeatBout, nSyl, sylLen, pauseLen, temperature, maleFemale, creakyBreathy, nonlinBalance,
     nonlinDep, jitterDep, jitterLen, vibratoFreq, vibratoDep, shimmerDep, attackLen, rolloff,
     rolloffOct, rolloffParab, rolloffParabHarm, rolloffKHz, rolloffLip, formantDep,
     formantDepStoch, vocalTract, subFreq, subDep, shortestEpoch, amDep, amFreq, amShape,
     samplingRate, windowLength, rolloffNoise) = [loc[p] for p in so.CHECKED_PARS]
    r_stream = hasattr(rng, 'rbinom1')     # R's own stream: every draw of the call comes from it
    if temperature > 0 and not r_stream:
        raise ValueError('temperature > 0 draws from R\'s stream: pass rng = oracle.rrng.RRng(seed)')

    pitchAnchors = _df(pitchAnchors)
    pitchAnchorsGlobal = _df(pitchAnchorsGlobal)
    amplAnchors = _df(amplAnchors)
    amplAnchorsGlobal = _df(amplAnchorsGlobal)
    mouthAnchors = _df(mouthAnchors)
    noiseAnchors = _df(noiseAnchors, t_hi=sylLen)
    if formants == 'default':
        formants = [f.copy() for f in DEFAULT_FORMANTS]
    elif formants is not None:
        formants = [np.array(f, dtype=np.float64) for f in formants]
    if formantsNoise is not None:
        formantsNoise = [np.array(f, dtype=np.float64) for f in formantsNoise]

    windowLength_points = math.floor(windowLength / 1000 * samplingRate / 2) * 2  # :317
    tempEffects = dict(sylLenDep=.02, formDrift=.3, formDisp=.2, pitchDriftDep=.5,
                       pitchDriftFreq=.125, pitchAnchorsDep=.05, noiseAnchorsDep=.1,
                       amplAnchorsDep=.1)

    if creakyBreathy < 0:  # :337-351
        nonlinBalance = min(100, nonlinBalance - creakyBreathy * 50)
        jitterDep = max(0, jitterDep - creakyBreathy / 2)
        shimmerDep = max(0, shimmerDep - creakyBreathy * 5)
        subDep = subDep * 2 ** (-creakyBreathy)
    elif creakyBreathy > 0:
        v = np.array([-120., -120.]) + creakyBreathy * 160
        v[v > so.PERMITTED['noiseAmpl'][2]] = so.PERMITTED['noiseAmpl'][2]
        noiseAnchors = (np.array([0., sylLen + 100]), v)
    rolloff = rolloff - creakyBreathy * 10  # :353-360
    rolloffOct = rolloffOct - creakyBreathy * 5
    subFreq = 2 * (subFreq - 50) / (1 + math.exp(-.1 * (50 - nonlinDep))) + 50
    jitterDep = 2 * jitterDep / (1 + math.exp(.1 * (50 - nonlinDep)))
    if maleFemale != 0:  # :364-379
        if pitchAnchors is not None:
            pitchAnchors = (pitchAnchors[0], pitchAnchors[1] * 2 ** maleFemale)
        if formants is not None:
            for f in formants:
                f[:, 1] = f[:, 1] * 1.25 ** maleFemale
        vocalTract = vocalTract * (1 - .25 * maleFemale)

    if r_stream:  # :394-400
        nSyl = int(math.floor(nSyl) + rng.rbinom1(1, nSyl - math.floor(nSyl)))
        repeatBout = int(math.floor(repeatBout) + rng.rbinom1(1, repeatBout - math.floor(repeatBout)))
    else:  # fraction 0: rbinom(1, 1, 0) draws nothing
        nSyl = int(math.floor(nSyl))
        repeatBout = int(math.floor(repeatBout))

    pars = dict(attackLen=attackLen, jitterDep=jitterDep, jitterLen=jitterLen,
                vibratoFreq=vibratoFreq, vibratoDep=vibratoDep, shimmerDep=shimmerDep,
                creakyBreathy=creakyBreathy, rolloff=rolloff, rolloffOct=rolloffOct,
                rolloffKHz=rolloffKHz, rolloffParab=rolloffParab,
                rolloffParabHarm=rolloffParabHarm, temperature=temperature,
                pitchDriftDep=tempEffects['pitchDriftDep'],
                pitchDriftFreq=tempEffects['pitchDriftFreq'], shortestEpoch=shortestEpoch,
                subFreq=subFreq, subDep=subDep, rolloffLip=rolloffLip, amDep=amDep,
                amFreq=amFreq, nonlinBalance=nonlinBalance, nonlinDep=nonlinDep,
                pitchFloor=pitchFloor, pitchCeiling=pitchCeiling,
                pitchSamplingRate=pitchSamplingRate, throwaway=throwaway,
                samplingRate=samplingRate, overlap=overlap)

    if (pitchAnchorsGlobal is not None and np.any(pitchAnchorsGlobal[1] != 0) and nSyl > 1):  # :448-462
        pitchDeltas = 2 ** (so.getSmoothContour(pitchAnchorsGlobal, length=nSyl,
                                                method='spline') / 12)
    else:
        pitchDeltas = np.ones(nSyl)

    if pitchAnchors is not None:  # :465-472
        t = pitchAnchors[0]
        if np.min(t) < 0:
            t = t - np.min(t)
        if np.max(t) > 1:
            t = t / np.max(t)
        pitchAnchors = (t, pitchAnchors[1])

    has_noise = noiseAnchors is not None and np.sum(noiseAnchors[1] > throwaway) > 0
    wiggleNoise = temperature > 0 and has_noise
    wiggleAmpl_per_syl = temperature > 0 and amplAnchors is not None and np.sum(amplAnchors[1] < -throwaway) > 0
    P = so.PERMITTED
    pars_to_vary = ['nonlinDep', 'attackLen', 'jitterDep', 'shimmerDep', 'rolloff', 'rolloffOct',
                    'shortestEpoch', 'subFreq', 'subDep']
    pars_to_round = ['attackLen', 'subFreq', 'subDep']
    bout = None
    for b in range(repeatBout):  # :482
        if temperature > 0:  # :484-506 (sd = 0 returns the mean without drawing)
            sylDur_s = sylLen
            if P['sylLen'][1] <= sylLen <= P['sylLen'][2]:
                sylDur_s = rnorm_bounded(rng, 1, sylLen, (P['sylLen'][2] - P['sylLen'][1]) * temperature *
                                         tempEffects['sylLenDep'], P['sylLen'][1], P['sylLen'][2])[0]
            pauseDur_s = rnorm_bounded(rng, 1, pauseLen, (P['pauseLen'][2] - P['pauseLen'][1]) * temperature *
                                       tempEffects['sylLenDep'], P['pauseLen'][1], P['pauseLen'][2])[0]
        else:
            sylDur_s = sylLen
            pauseDur_s = min(max(pauseLen, P['pauseLen'][1]), P['pauseLen'][2])
        if nSyl == 1:  # divideIntoSyllables, utilities_soundgen.R:515-551
            syllables = np.array([[0., sylDur_s]])
        else:
            rows = []
            c = 0.
            Td = temperature * tempEffects['sylLenDep']
            while len(rows) < nSyl:
                if Td > 0:
                    dur = rnorm_bounded(rng, 1, sylDur_s, sylDur_s * Td, P['sylLen'][1], P['sylLen'][2])[0]
                    pau = rnorm_bounded(rng, 1, pauseDur_s, pauseDur_s * Td, P['pauseLen'][1], P['pauseLen'][2])[0]
                else:
                    dur = min(max(sylDur_s, P['sylLen'][1]), P['sylLen'][2])
                    pau = min(max(pauseDur_s, P['pauseLen'][1]), P['pauseLen'][2])
                start = 1 + c
                end = start + dur
                rows.append([start, end])
                c = end + pau
            syllables = np.array(rows)
        syllableStartIdx = r_round(syllables[:, 0] * samplingRate / 1000)  # :517-532
        syllableStartIdx[0] = 1
        if noiseAnchors is not None and noiseAnchors[0][0] != 0:
            shift = -r_round(noiseAnchors[0][0] * samplingRate / 1000)
            if noiseAnchors[0][0] < 0:
                syllableStartIdx[0] = (syllableStartIdx - shift)[0]
            else:
                syllableStartIdx = syllableStartIdx - shift

        voiced = np.zeros(0)
        voiced_f0 = np.zeros(0)
        unvoiced = []
        for s in range(syllables.shape[0]):  # :540
            pars_syl = dict(pars)
            pitchAnchors_syl, amplAnchors_syl = pitchAnchors, amplAnchors
            if temperature > 0:  # :546-591
                for p in pars_to_vary:
                    lo_, hi_ = P[p][1], P[p][2]
                    pars_syl[p] = float(rnorm_bounded(rng, 1, pars[p], (hi_ - lo_) * temperature / 10, lo_, hi_,
                                                      roundToInteger=(p in pars_to_round))[0])
                if pitchAnchors_syl is not None:
                    pitchAnchors_syl = wiggleAnchors(rng, pitchAnchors_syl, temperature,
                                                     tempEffects['pitchAnchorsDep'], (0, P['pitch'][1]),
                                                     (1, P['pitch'][2]))
                if wiggleNoise:  # the result is overwritten at :646; only its draws matter
                    wiggleAnchors(rng, noiseAnchors, temperature, tempEffects['noiseAnchorsDep'],
                                  (-np.inf, P['noiseAmpl'][1]), (np.inf, P['noiseAmpl'][2]), wiggleAllRows=True)
                if wiggleAmpl_per_syl:
                    amplAnchors_syl = wiggleAnchors(rng, amplAnchors_syl, temperature,
                                                    tempEffects['amplAnchorsDep'], (0, 0), (1, -throwaway))
            dur_syl = float(syllables[s, 1] - syllables[s, 0])
            pitchContour_syl = None
            if pitchAnchors_syl is not None:
                pitchContour_syl = so.getSmoothContour(
                    pitchAnchors_syl, length=r_round(dur_syl * pitchSamplingRate / 1000),
                    samplingRate=pitchSamplingRate, valueFloor=pitchFloor,
                    valueCeiling=pitchCeiling, thisIsPitch=True,
                    method=contour_method) * pitchDeltas[s]
            if (dur_syl < so.PERMITTED['sylLen'][1]
                    or (noiseAnchors is not None and np.min(noiseAnchors[1]) >= 40)
                    or pitchAnchors_syl is None):
                syllable = np.zeros(int(r_round(dur_syl * samplingRate / 1000)))
                syl_f0 = syllable
            else:
                syllable, art = so.generateHarmonics(
                    pitchContour_syl, amplAnchors=amplAnchors_syl, rng=rng,
                    contour_method=contour_method, want_artefacts=True, **pars_syl)
                syl_f0 = syllable_track(art, samplingRate)
                assert syl_f0.size == syllable.size
            if s < syllables.shape[0] - 1:
                pause = np.zeros(int(math.floor((syllables[s + 1, 0] - syllables[s, 1]) *
                                                samplingRate / 1000)))
            else:
                pause = np.zeros(0)
            voiced = np.concatenate((voiced, syllable, pause))
            voiced_f0 = np.concatenate((voiced_f0, syl_f0, pause))

            if has_noise:  # :643-698
                t = noiseAnchors[0].copy()
                t[t > 0] = t[t > 0] * dur_syl / sylLen
                na_syl = (t, noiseAnchors[1])
                rng_t = float(np.max(t) - np.min(t))
                unvoicedDur_syl = int(r_round(rng_t * samplingRate / 1000))
                if formantsNoise is None:
                    spectralEnvelopeNoise = None
                else:
                    # :662 max(unlist(lapply(formantsNoise, length))) > 1 -- `length` of a
                    # formant (a list/data.frame of time, freq, amp, width) is 4, so the
                    # test is TRUE for any formantsNoise list: noise formants always "move"
                    moving = True
                    nInt = int(r_round(rng_t / 10)) if moving else 1
                    spectralEnvelopeNoise = so.getSpectralEnvelope(
                        nr=windowLength_points / 2, nc=nInt, formants=formantsNoise,
                        formantDep=formantDep, rolloffLip=rolloffLip, mouthAnchors=mouthAnchors,
                        temperature=temperature, samplingRate=samplingRate,
                        vocalTract=vocalTract, contour_method=contour_method,
                        formDrift=tempEffects['formDrift'], formDisp=tempEffects['formDisp'],
                        formantDepStoch=formantDepStoch, rng=rng)
                unvoiced.append(so.generateNoise(
                    length=unvoicedDur_syl, noiseAnchors=na_syl, rolloffNoise=rolloffNoise,
                    attackLen=attackLen, samplingRate=samplingRate,
                    windowLength_points=windowLength_points, overlap=overlap,
                    throwaway=throwaway, filterNoise=spectralEnvelopeNoise, rng=rng,
                    contour_method=contour_method))

        sound = voiced  # :708-714
        sound_f0 = voiced_f0
        if len(unvoiced) > 0 and formantsNoise is None:
            for s in range(len(unvoiced)):
                sound = so.addVectors(sound, unvoiced[s], insertionPoint=syllableStartIdx[s])
                sound_f0 = so.addVectors(sound_f0, np.zeros(len(unvoiced[s])), insertionPoint=syllableStartIdx[s])

        if amplAnchorsGlobal is not None and np.sum(amplAnchorsGlobal[1] < -throwaway) > 0:  # :721-733
            ag = (amplAnchorsGlobal[0], 2 ** (amplAnchorsGlobal[1] / 10))
            amplEnvelope = so.getSmoothContour(ag, length=sound.size, valueFloor=0,
                                               valueCeiling=-throwaway,
                                               samplingRate=samplingRate, method=contour_method)
            sound = sound * amplEnvelope
            amplAnchorsGlobal = ag  # the reference overwrites the anchors in place (:724)

        if r_sum(sound) == 0:  # :736-739
            soundFiltered = sound
        else:
            windowLength_points = min(windowLength_points, math.floor(sound.size / 2))  # :743
            step = so.frame_starts(sound.size, windowLength_points, overlap)
            nc = step.size
            nr = windowLength_points / 2
            if formants is not None:  # :751-758
                # max(sapply(formants, function(x) sapply(x, length))) > 1
                movingFormants = max(f.shape[0] for f in formants) > 1
            else:
                movingFormants = False
            if mouthAnchors is not None and np.sum(mouthAnchors[1] != .5) > 0:
                movingFormants = True
            nInt = nc if movingFormants else 1
            spectralEnvelope = so.getSpectralEnvelope(
                nr=nr, nc=nInt, formants=formants, formantDep=formantDep, rolloffLip=rolloffLip,
                mouthAnchors=mouthAnchors, temperature=temperature, samplingRate=samplingRate,
                vocalTract=vocalTract, contour_method=contour_method, formDrift=tempEffects['formDrift'],
                formDisp=tempEffects['formDisp'], formantDepStoch=formantDepStoch, rng=rng)
            soundFiltered = so.filter_sound(sound, spectralEnvelope, windowLength_points, overlap)

        filtered_f0 = np.zeros(soundFiltered.size)
        m = min(soundFiltered.size, sound_f0.size)
        filtered_f0[:m] = sound_f0[:m]
        if len(unvoiced) > 0 and formantsNoise is not None:  # :813-818
            for s in range(len(unvoiced)):
                soundFiltered = so.addVectors(soundFiltered, unvoiced[s],
                                              insertionPoint=syllableStartIdx[s])
                filtered_f0 = so.addVectors(filtered_f0, np.zeros(len(unvoiced[s])),
                                            insertionPoint=syllableStartIdx[s])
        if amDep > 0:  # :821-833
            sig = so.getSigmoid(length=soundFiltered.size, samplingRate=samplingRate,
                                freq=amFreq, shape=amShape)
            soundFiltered = soundFiltered * (1 - sig * amDep / 100)
        if b == 0:  # :836-842
            bout = soundFiltered
            bout_f0 = filtered_f0
        else:
            bout = np.concatenate((bout, np.zeros(int(pauseLen * samplingRate / 1000)),
                                   soundFiltered))
            bout_f0 = np.concatenate((bout_f0, np.zeros(int(pauseLen * samplingRate / 1000)), filtered_f0))
    if addSilence is not None:  # :846-849
        n = int(r_round(samplingRate / 1000 * addSilence))
        bout = np.concatenate((np.zeros(n), bout, np.zeros(n)))
        bout_f0 = np.concatenate((np.zeros(n), bout_f0, np.zeros(n)))
    assert bout_f0.size == bout.size
    return bout, bout_f0
