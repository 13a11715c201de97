"""Pins the plain-C oracle (oracle/maxi_oracle.c) BIT-FOR-BIT against the unmodified reference
compiled by oracle/Makefile (oracle/_ref/libmaxiref.so).

CPU only. Each test drives one library through a scenario (run(kind)); the port's values must equal the
reference's, live where the compiled reference is present and against its stored trace everywhere
(tests/reference_trace.py).
Tolerance: none. fp64 and fp32 values are compared with ==, integer state exactly.
"""
import itertools

import numpy as np
import pytest

from maximilian_b200 import workloads as W

OSCS = ["sinewave", "coswave", "phasor", "saw", "square", "pulse", "impulse", "triangle", "phasorbetween"]
FILTS = ["none", "lores", "hires", "svf", "biquad"]


_configure = W.configure_bank


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize("osc,filt", list(itertools.product(OSCS, FILTS)))
def test_osc_filter_chains_bit_exact(port, reference, osc, filt):
    def run(kind):
        V, B = 37, 257
        p = W.voice_params(V, seed=11)
        b = port.Bank(V, kind=kind, osc=osc, filt=filt)
        _configure(b, filt, p, False, False)
        for blk in range(3):                      # state carried over consecutive blocks
            o, m = b.process(B, want_mix=True)
            yield f"out {blk}", o
            yield f"mix {blk}", m
        for s in ("phase", "filt0", "filt1", "filt2"):
            yield s, b.get(s)
    reference.check(run)


@pytest.mark.parametrize("btype", ["lowpass", "highpass", "bandpass", "notch", "peak", "lowshelf", "highshelf"])
@pytest.mark.parametrize("gain_sign", [1.0, -1.0])
def test_biquad_types_bit_exact(port, reference, btype, gain_sign):
    def run(kind):
        V, B = 16, 300
        p = W.voice_params(V, seed=5)
        p["gain"] = gain_sign * (0.5 + 11.5 * np.random.default_rng(3).random(V))
        b = port.Bank(V, kind=kind, osc="saw", filt="biquad", biquad_type=btype)
        _configure(b, "biquad", p, False, False)
        yield "out", b.process(B)[0]
    reference.check(run)


@pytest.mark.parametrize("mix", [(1, 0, 0, 0), (0, 1, 0, 0), (0, 0, 1, 0), (0, 0, 0, 1), (0.3, 0.2, 0.4, 0.1)])
def test_svf_mixes_bit_exact(port, reference, mix):
    def run(kind):
        V, B = 16, 300
        p = W.voice_params(V, seed=6)
        p["res_svf"][0] = 0.0                     # res == 0 -> damping 0 branch (src/maximilian.h:1327)
        b = port.Bank(V, kind=kind, osc="saw", filt="svf", svf_mix=tuple(float(m) for m in mix))
        _configure(b, "svf", p, False, False)
        yield "out", b.process(B)[0]
    reference.check(run)


def test_lores_clamps_bit_exact(port, reference):
    # cutoff < 10 -> 10, cutoff > sr -> sr (NaN: z == 1 gives 0/0), resonance < 1 -> 1  (SURVEY.md A3)
    def run(kind):
        V, B = 6, 64
        p = W.voice_params(V, seed=2)
        p["cutoff"] = np.array([1.0, 9.999, 10.0, 47999.0, 48000.0, 96000.0])
        p["q_lores"] = np.array([0.0, 0.5, 1.0, 1.5, 2.0, 3.0])
        for filt in ("lores", "hires"):
            b = port.Bank(V, kind=kind, osc="saw", filt=filt)
            _configure(b, filt, p, False, False)
            o, _ = b.process(B)
            if kind == "port":
                assert np.isnan(o[-1, 4]) and np.isnan(o[-1, 5])
            yield filt, o
    reference.check(run)


def test_sample_rates(port, reference):
    def run(kind):
        for sr in (44100, 48000, 96000):
            V, B = 8, 200
            p = W.voice_params(V, seed=sr)
            b = port.Bank(V, kind=kind, osc="sinewave", filt="svf", sample_rate=sr)
            _configure(b, "svf", p, False, False)
            yield f"out {sr}", b.process(B)[0]
    reference.check(run)


@pytest.mark.parametrize("filt", ["none", "lores"])
def test_env_state_machine_bit_exact(port, reference, filt):
    def run(kind):
        V, B = 64, 512
        p = W.voice_params(V, seed=9)
        p["env_holdtime"] = np.array([1, 1, 0, 5, 100, 1000, 1, 3] * (V // 8), dtype=np.float64)
        b = port.Bank(V, kind=kind, osc="saw", filt=filt, env=True)
        _configure(b, filt, p, True, False)
        for blk in range(8):
            on, off = W.gate(V, B, blk)
            if blk == 5:                          # retrigger while still releasing, gate across the whole block
                on[:] = 0; off[:] = B
            yield f"out {blk}", b.process(B, on, off)[0]
            for s in ("env_amplitude", "env_output", "env_holdcount", "env_flags"):
                yield f"{s} {blk}", b.get(s)
    reference.check(run)


def test_env_setters(port, reference):
    def run(kind):
        lib = port.load(kind)
        for ms in (0.5, 1.0, 2.0, 17.3, 500.0):
            for sr in (44100, 48000):
                yield f"attack {ms} {sr}", lib.mxo_env_attack_coeff(ms, sr)
                yield f"attack_ms {ms} {sr}", lib.mxo_env_attack_ms_coeff(ms, sr)
                yield f"decay {ms} {sr}", lib.mxo_env_decay_coeff(ms, sr)
        p = W.voice_params(8, seed=1)
        if kind == "port":
            att, dec, rel = W.env_coeffs(p)       # math.pow == libm pow
        else:
            att = [lib.mxo_env_attack_coeff(p["attack_ms"][i], 48000) for i in range(8)]
            dec = [lib.mxo_env_decay_coeff(p["decay_ms"][i], 48000) for i in range(8)]
            rel = [lib.mxo_env_decay_coeff(p["release_ms"][i], 48000) for i in range(8)]
        for i in range(8):
            yield f"env_coeffs {i}", np.array([att[i], dec[i], rel[i]], dtype=np.float64)
    reference.check(run)


def test_delayline_indices_and_ring_bit_exact(port, reference):
    def run(kind):
        # small V: every reference maxiDelayline is a 5.6 MB object (src/maximilian.h:273)
        V, B, cap = 12, 700, 512
        p = W.voice_params(V, seed=4, delay_size=cap, ragged_delay=True)
        p["delay_size"][:4] = [1, 2, 3, cap]
        b = port.Bank(V, kind=kind, osc="saw", env=True, delay=True, delay_capacity=cap)
        _configure(b, "none", p, True, True)
        for blk in range(4):
            on, off = W.gate(V, B, blk)
            if blk == 2:                          # size shrinks mid-stream: phase >= size -> 0 on the next call (A6)
                p["delay_size"] = np.maximum(1, p["delay_size"] // 2)
                b.set("delay_size", p["delay_size"])
            yield f"out {blk}", b.process(B, on, off)[0]
            yield f"delay_phase {blk}", b.get("delay_phase")     # integer index: exact
        for v in range(V):
            yield f"ring {v}", b.ring(v, cap)
    reference.check(run)


def fm_frequencies(V, B, blk, seed=5):
    """freq[t][v] = carrier + depth * sin(2*pi*rate*t/sr): what 5.FM1's play() feeds its carrier (main.cpp:29)."""
    rng = np.random.default_rng(seed)
    carrier = 110.0 * np.exp2(3.0 * rng.random(V)); depth = 50.0 * rng.random(V); rate = 0.5 + 8.0 * rng.random(V)
    t = (blk * B + np.arange(B))[:, None] / 48000.0
    return carrier[None, :] + depth[None, :] * np.sin(2 * np.pi * rate[None, :] * t)


@pytest.mark.parametrize("osc,filt", [("sinewave", "none"), ("saw", "svf"), ("triangle", "lores")])
def test_per_sample_frequency_bit_exact(port, reference, osc, filt):
    def run(kind):
        V, B = 21, 200
        p = W.voice_params(V, seed=31)
        b = port.Bank(V, kind=kind, osc=osc, filt=filt)
        _configure(b, filt, p)
        for blk in range(3):
            yield f"out {blk}", b.process(B, freq_tv=fm_frequencies(V, B, blk))[0]
        yield "out block-constant", b.process(B)[0]           # back to the block-constant frequency
    reference.check(run)


def cutoff_sweeps(V, B, blk, seed=6):
    """cutoff[t][v] = centre * 2^(depth * sin(2*pi*rate*t/sr)): an LFO-swept filter, 60 Hz .. 12 kHz."""
    rng = np.random.default_rng(seed)
    centre = 200.0 * np.exp2(4.0 * rng.random(V)); depth = 1.5 * rng.random(V); rate = 0.2 + 6.0 * rng.random(V)
    t = (blk * B + np.arange(B))[:, None] / 48000.0
    return centre[None, :] * np.exp2(depth[None, :] * np.sin(2 * np.pi * rate[None, :] * t))


@pytest.mark.parametrize("osc,filt,fm", [("saw", "svf", False), ("saw", "lores", False), ("phasor", "hires", True), ("square", "svf", True)])
def test_per_sample_cutoff_bit_exact(port, reference, osc, filt, fm):
    # lores/hires take the cutoff per call; the SVF patch calls setCutoff() per sample (src/maximilian.h:1287-1290)
    def run(kind):
        V, B = 19, 160
        p = W.voice_params(V, seed=33)
        b = port.Bank(V, kind=kind, osc=osc, filt=filt)
        _configure(b, filt, p)
        for blk in range(3):
            cu = cutoff_sweeps(V, B, blk); f = fm_frequencies(V, B, blk) if fm else None
            o, m = b.process(B, freq_tv=f, cutoff_tv=cu, want_mix=True)
            yield f"out {blk}", o
            yield f"mix {blk}", m
        yield "out block-constant", b.process(B)[0]           # the block-constant cutoff is in force again
        for s in ("filt0", "filt1"):
            yield s, b.get(s)
    reference.check(run)


def test_per_sample_cutoff_not_for_biquad(port, reference):
    def run(kind):
        bq = port.Bank(4, osc="saw", filt="biquad", kind=kind)
        bq.set("cutoff", 800.0); bq.set("resonance", 1.0); bq.set("gain", 0.0)
        with pytest.raises(RuntimeError):
            bq.process(8, cutoff_tv=np.full((8, 4), 500.0))
        yield "refused", True
    reference.check(run)


def flanger_sizes(V, B, blk, cap, seed=7):
    """size[t][v] = delay + triangle-ish LFO * depth * delay + 1, like maxiFlanger::flange feeds dl() (src/maximilian.h:1144-1180);
    some voices sweep down to 1 slot, some stay constant; every value <= cap."""
    rng = np.random.default_rng(seed)
    delay = rng.integers(8, cap // 2, V).astype(np.float64); depth = rng.random(V); rate = 0.5 + 20.0 * rng.random(V)
    depth[::5] = 0.0
    t = (blk * B + np.arange(B))[:, None] / 48000.0
    lfo = 2.0 * np.abs(2.0 * ((rate[None, :] * t) % 1.0) - 1.0) - 1.0
    return np.clip(np.floor(delay[None, :] + lfo * depth[None, :] * delay[None, :] + 1.0), 1, cap)


@pytest.mark.parametrize("delay", ["dl", "position"])
def test_per_sample_delay_size_bit_exact(port, reference, delay):
    def run(kind):
        V, B, cap = 10, 300, 256            # small V: every reference maxiDelayline is a 5.6 MB object
        p = W.voice_params(V, seed=41, delay_size=cap, ragged_delay=True)
        b = port.Bank(V, kind=kind, osc="saw", filt="lores", env=True, delay=delay, delay_capacity=cap)
        _configure(b, "lores", p, True, True)
        if delay == "position":
            b.set("delay_position", np.arange(V, dtype=np.float64) * 3.0)
        for blk in range(3):
            on, off = W.gate(V, B, blk)
            yield f"out {blk}", b.process(B, on, off, delay_size_tv=flanger_sizes(V, B, blk, cap))[0]
            yield f"delay_phase {blk}", b.get("delay_phase")
        yield "out block-constant", b.process(B)[0]           # back to the block-constant size
        for v in range(V):
            yield f"ring {v}", b.ring(v, cap)
    reference.check(run)


def test_env_ar_bit_exact(port, reference):
    # maxiEnv::ar(input, attack, release, holdtime, trigger), src/maximilian.cpp:1319-1358
    def run(kind):
        V, B = 48, 400
        p = W.voice_params(V, seed=19)
        att, dec, rel = W.env_coeffs(p)
        hold = np.array([1, 0, 5, 50, 300, 1, 2, 1000] * (V // 8), dtype=np.float64)
        b = port.Bank(V, kind=kind, osc="saw", filt="lores", env="ar")
        _configure(b, "lores", p)
        b.set("env_attack", att); b.set("env_release", rel); b.set("env_holdtime", hold)
        for blk in range(6):
            on, off = W.gate(V, B, blk)
            if blk == 3:
                on[:] = 0; off[:] = B
            yield f"out {blk}", b.process(B, on, off)[0]
            for s in ("env_amplitude", "env_output", "env_holdcount", "env_flags"):
                yield f"{s} {blk}", b.get(s)
    reference.check(run)


def test_dl_from_position_bit_exact(port, reference):
    # maxiDelayline::dlFromPosition, src/maximilian.cpp:431-439
    def run(kind):
        V, B, cap = 10, 300, 256
        p = W.voice_params(V, seed=23, delay_size=cap, ragged_delay=True)
        pos = np.array([0, 1, 5, 63, 64, 100, 200, 255, 300, 17], dtype=np.float64)     # 300 >= size -> 0
        b = port.Bank(V, kind=kind, osc="saw", delay="position", delay_capacity=cap)
        _configure(b, "none", p, False, True)
        b.set("delay_position", pos)
        for blk in range(3):
            yield f"out {blk}", b.process(B)[0]
            yield f"delay_phase {blk}", b.get("delay_phase")
        for v in range(V):
            yield f"ring {v}", b.ring(v, cap)
    reference.check(run)


def test_delay_size_nonpositive(port, reference):
    def run(kind):
        V, B = 3, 20
        b = port.Bank(V, kind=kind, osc="saw", delay=True, delay_capacity=16)
        b.set("freq", [100.0, 200.0, 300.0]); b.set("delay_size", [0.0, -3.0, 1.0]); b.set("delay_feedback", 0.7)
        yield "out", b.process(B)[0]
        yield "delay_phase", b.get("delay_phase")
    reference.check(run)


def test_threaded_partition_matches_serial(port):
    V, B = 64, 128
    p = W.voice_params(V, seed=3)
    a = port.Bank(V, osc="saw", filt="biquad"); b = port.Bank(V, osc="saw", filt="biquad")
    _configure(a, "biquad", p, False, False); _configure(b, "biquad", p, False, False)
    oa, ma = a.process(B, want_mix=True, threads=1)
    ob, mb = b.process(B, want_mix=True, threads=4)
    assert _same(oa, ob)
    np.testing.assert_allclose(ma, mb, rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------ spectral

@pytest.mark.parametrize("n,hop", [(1024, 512), (1024, 256), (512, 128), (256, 256), (64, 16)])
def test_stft_bit_exact(port, reference, n, hop):
    def run(kind):
        C = 5
        x = W.channel_streams(C, 6 * n + 37, seed=n + hop)
        x[1] *= 1000.0
        x[2] = 0.0
        s = port.Stft(C, n, hop, kind=kind)
        yield "window", s.window()
        # feed in uneven chunks: the frame schedule (integer pos) must agree exactly
        cuts = [0, 3, hop - 1, hop, 2 * n + 5, x.shape[1]]
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            r = s.process(x[:, lo:hi])
            for k in ("re", "im", "mags", "phases"):
                yield f"{k} {lo}:{hi}", r[k]
    reference.check(run)


def test_stft_frame_schedule(port):
    # first frame after hop samples; 93 frames in 48000 samples at hop 512 (SURVEY.md section 4, item 4)
    s = port.Stft(1, 1024, 512)
    r = s.process(np.zeros((1, 48000), dtype=np.float32))
    assert r["mags"].shape[1] == 93
    s = port.Stft(1, 1024, 512)
    assert s.process(np.zeros((1, 511), dtype=np.float32))["mags"].shape[1] == 0
    assert s.process(np.zeros((1, 1), dtype=np.float32))["mags"].shape[1] == 1


@pytest.mark.parametrize("cfg", [(512, 42, 40, 20.0, 20000.0, 48000), (512, 42, 13, 20.0, 20000.0, 44100),
                                 (512, 256, 13, 20.0, 20000.0, 48000), (256, 20, 12, 100.0, 8000.0, 48000)])
def test_mfcc_bit_exact(port, reference, cfg):
    bins = cfg[0]
    st = port.Stft(3, 2 * bins, bins)
    mags = st.process(W.channel_streams(3, 2 * bins * 8, seed=bins))["mags"]
    mags[0, 0] = 0.0                                   # silent frame: log gate (> 1e-6) takes the 0 branch

    def run(kind):
        c, m = port.Mfcc(*cfg, kind=kind).process(mags)
        if kind == "port":
            assert np.all(m[..., 0] == 0.0)            # filter 0 is never initialised by the reference (A13)
        yield "melbands", m
        yield "coeffs", c
    reference.check(run)


def test_spectral_features_bit_exact(port, reference):
    # maxiFFT::magsToDB / spectralFlatness / spectralCentroid, src/libs/maxiFFT.cpp:101-132
    mags = port.Stft(3, 1024, 512).process(W.channel_streams(3, 8192, seed=8))["mags"]
    mags[0, 0] = 0.0                                  # all-zero frame: both features return 0
    mags[1, 1, :7] = 0.0                              # zeros are skipped by the geometric mean

    def run(kind):
        for sr in (44100, 48000):
            for name, x in zip(("db", "flatness", "centroid"), port.spectral_features(mags, 1024, sr, kind=kind)):
                yield f"{name} {sr}", x
    reference.check(run)


@pytest.mark.parametrize("n,hop", [(1024, 512), (1024, 256), (256, 64)])
def test_istft_bit_exact(port, reference, n, hop):
    C = 3
    x = W.channel_streams(C, 10 * n, seed=77)
    r = port.Stft(C, n, hop).process(x)

    def run(kind):
        s = port.Istft(C, n, hop, kind=kind)
        F = r["mags"].shape[1]
        for lo, hi in ((0, 3), (3, F)):
            yield f"y {lo}:{hi}", s.process(r["mags"][:, lo:hi], r["phases"][:, lo:hi])
    reference.check(run)


# ---- maxiFFTOctaveAnalyzer / maxiBark (SURVEY.md 8f-3) ------------------------------------------------------------------------

@pytest.mark.parametrize("per_octave,sr", [(1, 48000), (3, 48000), (3, 44100), (6, 48000), (0, 48000)])
def test_octave_analyser_port_equals_reference(port, reference, per_octave, sr):
    """maxiFFTOctaveAnalyzer::setup + calculate per channel (float sums in bin order, peak hold / decay carried across frames and
    calls), with the public members changed from their defaults: averages and peaks bit for bit."""
    x = W.channel_streams(3, 1024 * 9, seed=5)
    mags = port.Stft(3, 1024, 512, kind="port").process(x)["mags"]

    def run(kind):
        a = port.Octave(3, sr, 512, per_octave, kind=kind)
        assert a.n_averages > 0
        yield "n_averages", a.n_averages
        a.config(2, 0.8, 1.0, 0.01)
        for lo, hi in ((0, 5), (5, mags.shape[1])):
            av, pk = a.process(mags[:, lo:hi])
            yield f"averages {lo}:{hi}", av
            yield f"peaks {lo}:{hi}", pk
    reference.check(run)


@pytest.mark.parametrize("sr,bs", [(48000, 1024), (44100, 1024), (48000, 512), (22050, 256)])
def test_bark_port_equals_reference(port, reference, sr, bs):
    """maxiBarkScaleAnalyser: integer binToHz, int band ends, the 25th band limit written behind bbLimits[24] -- specific, relative and
    total loudness bit for bit (the reference class is compiled at -O0 inside the shim: its setup() is undefined behaviour that -O2
    turns into a crash)."""
    x = W.channel_streams(3, 1024 * 9, seed=6)
    mags = np.ascontiguousarray(port.Stft(3, 1024, 512, kind="port").process(x)["mags"][..., :bs // 2])
    pa = port.bark(mags, sr, bs, "port")
    assert np.all(pa[1].max(axis=-1) == 1.0)

    def run(kind):
        for name, u in zip(("specific", "relative", "total"), pa if kind == "port" else port.bark(mags, sr, bs, kind)):
            yield name, u
    reference.check(run)


@pytest.mark.parametrize("filt,delay,env", [("none", False, "adsr"), ("lores", False, "ar"), ("svf", True, "adsr")])
def test_per_sample_trigger_port_equals_reference(port, reference, filt, delay, env):
    """maxiEnv::trigger written on every sample (mxo_bank_process_mod2): several notes per block, both envelope kinds."""
    def run(kind):
        rng = np.random.default_rng(5)
        V, B, cap = 12, 400, 64
        p = W.voice_params(V, seed=61, delay_size=cap, ragged_delay=True)
        b = port.Bank(V, osc="saw", filt=filt, env=env, delay=delay, delay_capacity=cap, kind=kind)
        W.configure_bank(b, filt, p, env=True, delay=delay)
        for blk in range(3):
            tv = (rng.random((B, V)) < 0.5).astype(np.uint8)
            tv[:, 0] = 0; tv[:, 1] = 1
            tv[100:250, 2:6] = 1; tv[250:260, 2:6] = 0; tv[260:300, 2:6] = 1
            o, m = b.process(B, trig_tv=tv, want_mix=True)
            yield f"out {blk}", o
            yield f"mix {blk}", m
            for s_ in ("env_holdcount", "env_flags", "env_amplitude", "env_output"):
                yield f"{s_} {blk}", b.get(s_)
    reference.check(run)


@pytest.mark.parametrize("osc,filt,env,cm,dsz", [("saw", "none", True, False, False), ("saw", "lores", True, True, False), ("pulse", "svf", False, True, False),
                                                 ("phasorbetween", "biquad", True, False, False), ("sinewave", "hires", False, True, True)])
def test_modulated_chain_with_a_delay_line_port_equals_reference(port, reference, osc, filt, env, cm, dsz):
    """Per-sample frequency / cutoff (/ delay size / trigger) on a chain that ends in maxiDelayline::dl -- the combinations the modulated
    instantiation of K2 is tested against (tests/test_gpu_bank.py::test_modulated_frequency_and_cutoff_with_a_delay_line compares it
    with the port): the port itself against the compiled reference, samples, ring index and ring contents bit for bit."""
    def run(kind):
        V, B, cap = 23, 150, 96
        p = W.voice_params(V, seed=61, delay_size=cap, ragged_delay=True)
        b = port.Bank(V, kind=kind, osc=osc, filt=filt, env=env, delay=True, delay_capacity=cap)
        _configure(b, filt, p, env, True)
        rng = np.random.default_rng(8)
        for blk in range(3):
            f = fm_frequencies(V, B, blk); cu = cutoff_sweeps(V, B, blk) if cm else None
            tv = (rng.random((B, V)) < 0.4).astype(np.uint8) if env else None
            sz = np.floor(1 + (cap - 1) * rng.random((B, V))) if dsz else None
            o, m = b.process(B, freq_tv=f, cutoff_tv=cu, trig_tv=tv, delay_size_tv=sz, want_mix=True)
            yield f"out {blk}", o
            yield f"mix {blk}", m
            yield f"delay_phase {blk}", b.get("delay_phase")
        on, off = (W.gate(V, B, 3) if env else (None, None))
        yield "out gated", b.process(B, on, off)[0]
        for v in (0, V // 2, V - 1):
            yield f"ring {v}", b.ring(v, cap)
    reference.check(run)


def test_per_sample_analysis_resynthesis_idiom(port, reference):
    """`if (fft.process(sample)) ...; out = ifft.process(fft.getMagnitudes(), fft.getPhases())` on every sample, run by the compiled
    reference (ref_shim: mxo_ref_per_sample_roundtrip), equals the block functions composed the way the C++ layer's per-sample signatures
    compose them (tests/test_cpp_dropin.py::test_per_sample_feature_extractor_matches_oracle): a frame fires on the last sample of every
    hop; the resynthesis reads zeros during the first hop and frame k - 1 during hop k. Bit for bit."""
    import ctypes as C
    N, n, hop, bins = 6 * 1024 + 300, 1024, 512, 512
    x = W.channel_streams(1, N, seed=45)

    def run(kind):
        if kind == "reference":
            fn = port.load("reference").mxo_ref_per_sample_roundtrip
            fn.restype = C.c_int32
            fn.argtypes = [C.POINTER(C.c_float), C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_uint8)]
            y = np.empty(N, dtype=np.float32); fired = np.empty(N, dtype=np.uint8)
            F = fn(x.ctypes.data_as(C.POINTER(C.c_float)), N, n, hop, y.ctypes.data_as(C.POINTER(C.c_float)), fired.ctypes.data_as(C.POINTER(C.c_uint8)))
            yield "frames", F
            yield "fired", np.nonzero(fired)[0]
            yield "y", y
            return
        F = N // hop
        yield "frames", F
        yield "fired", hop * np.arange(1, F + 1) - 1
        o = port.Stft(1, n, hop, kind="port").process(x)
        K = (N + hop - 1) // hop
        z = np.zeros((1, 1, bins), dtype=np.float32)
        oy = port.Istft(1, n, hop, kind="port").process(np.concatenate([z, o["mags"][:, :K - 1]], axis=1), np.concatenate([z, o["phases"][:, :K - 1]], axis=1))
        yield "y", oy[0, :N]
    reference.check(run)
