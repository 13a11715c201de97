"""Randomised pin of the plain-C oracle against the compiled reference: chains, sizes, sample rates and parameter
values drawn from seeded generators -- including the ugly corners (zero / negative / above-Nyquist frequencies, duty
outside [0, 1], resonance 0, hold times 0, one-slot delay lines, gates that open and close inside one block, modulated
arguments) -- compared BIT FOR BIT over consecutive blocks, state included. CPU only; against the stored trace of the
reference everywhere and the compiled reference itself where it is built (tests/reference_trace.py).
"""
import numpy as np
import pytest

from maximilian_b200 import workloads as W

OSCS = ["sinewave", "coswave", "phasor", "saw", "square", "pulse", "impulse", "triangle", "phasorbetween"]
FILTS = ["none", "lores", "hires", "svf", "biquad"]
BQ = ["lowpass", "highpass", "bandpass", "notch", "peak", "lowshelf", "highshelf"]
RATES = [8000, 22050, 44100, 48000, 96000]


def _draw(seed):
    rng = np.random.default_rng(1000 + seed)
    c = dict(osc=OSCS[rng.integers(len(OSCS))], filt=FILTS[rng.integers(len(FILTS))], sr=RATES[rng.integers(len(RATES))],
             env=[False, True, "ar"][rng.integers(3)], delay=[False, True, "position"][rng.integers(3)],
             V=int(rng.integers(1, 10)), B=int(rng.integers(1, 160)), cap=int(rng.integers(1, 80)),
             bq=BQ[rng.integers(len(BQ))], mix=tuple(np.round(rng.random(4), 2)) if rng.random() < 0.5 else (1.0, 0.0, 0.0, 0.0))
    V = c["V"]
    p = W.voice_params(V, seed=seed, delay_size=c["cap"], ragged_delay=True)
    nyq = c["sr"] / 2
    # corners, a few voices each
    p["freq"][rng.random(V) < 0.15] = 0.0
    p["freq"][rng.random(V) < 0.10] *= -1.0
    p["freq"][rng.random(V) < 0.10] = nyq * 1.7
    p["duty"][rng.random(V) < 0.2] = rng.choice([-0.3, 0.0, 1.0, 1.4])
    p["cutoff"] = np.minimum(p["cutoff"], 0.45 * c["sr"])           # lores at fc == sr is NaN by design (SURVEY.md A3): covered elsewhere
    p["cutoff"][rng.random(V) < 0.15] = 5.0                          # below the lores clamp
    p["res_svf"][rng.random(V) < 0.2] = 0.0                          # maxiSVF: damping 0 branch
    p["q_lores"][rng.random(V) < 0.2] = 0.2                          # below the lores clamp
    p["gain"] = np.round(rng.uniform(-15, 15, V), 1)
    p["env_holdtime"] = rng.choice([0.0, 1.0, 2.0, 7.0, 300.0], V)
    p["delay_size"] = np.minimum(p["delay_size"], c["cap"])
    p["delay_size"][rng.random(V) < 0.2] = 1.0
    p["delay_feedback"][rng.random(V) < 0.1] = 0.0
    p["pan"][rng.random(V) < 0.2] = rng.choice([-0.5, 0.0, 1.0, 1.5])
    p["phasor_start"][rng.random(V) < 0.2] = 0.9                     # start above end: the ramp never advances past `start`
    return c, p, rng


@pytest.mark.parametrize("seed", range(60))
def test_random_chain_bit_exact(port, reference, seed):
    def run(kind):
        c, p, rng = _draw(seed)
        V, B = c["V"], c["B"]
        kw = dict(osc=c["osc"], filt=c["filt"], env=c["env"], delay=c["delay"], sample_rate=c["sr"], biquad_type=c["bq"],
                  svf_mix=tuple(float(m) for m in c["mix"]), delay_capacity=c["cap"])
        b = port.Bank(V, kind=kind, **kw)
        W.configure_bank(b, c["filt"], p, bool(c["env"]), bool(c["delay"]), sample_rate=c["sr"])
        if c["delay"] == "position":
            b.set("delay_position", np.minimum(np.arange(V) * 2.0, c["cap"] - 1))
        mod_ok = not c["env"] and not c["delay"]
        for blk in range(3):
            on = rng.integers(0, B + 1, V).astype(np.int32); off = rng.integers(0, B + 2, V).astype(np.int32)
            kwp = {}
            if mod_ok and blk == 1:
                kwp["freq_tv"] = 50.0 + 2000.0 * rng.random((B, V))
                if c["filt"] in ("lores", "hires", "svf"):
                    kwp["cutoff_tv"] = 30.0 + 0.4 * c["sr"] * rng.random((B, V))
            if c["delay"] and blk == 1:
                kwp["delay_size_tv"] = rng.integers(1, c["cap"] + 1, (B, V)).astype(np.float64)
            o, m = b.process(B, on, off, want_mix=True, **kwp)
            yield f"out {blk} {c}", o
            yield f"mix {blk} {c}", m
        states = ["phase", "filt0", "filt1"] + (["filt2"] if c["filt"] == "svf" else [])
        if c["env"]:
            states += ["env_amplitude", "env_output", "env_holdcount", "env_flags"]
        if c["delay"]:
            states += ["delay_phase"]
        for s in states:
            yield f"{s} {c}", b.get(s)
        if c["delay"]:
            for v in range(V):
                yield f"ring {v} {c}", b.ring(v, c["cap"])
    reference.check(run)


@pytest.mark.parametrize("seed", range(12))
def test_random_spectral_bit_exact(port, reference, seed):
    def run(kind):
        rng = np.random.default_rng(5000 + seed)
        n = int(rng.choice([64, 128, 256, 512, 1024, 2048]))
        hop = int(rng.choice([n // 8, n // 4, n // 2, n]))
        C = int(rng.integers(1, 4))
        x = W.channel_streams(C, int(rng.integers(n, 6 * n)), seed=seed)
        x[0] *= float(rng.choice([1e-6, 1.0, 1e4]))
        s = port.Stft(C, n, hop, kind=kind)
        cuts = np.unique(np.r_[0, rng.integers(0, x.shape[1], 3), x.shape[1]])
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            r = s.process(x[:, lo:hi])
            for k in ("mags", "phases", "re", "im"):
                yield f"{k} {lo}:{hi} (n {n}, hop {hop})", r[k]
        if n >= 128:
            nf, nc = int(rng.integers(8, 43)), int(rng.integers(4, 41))
            mf = port.Mfcc(n // 2, nf, nc, 20.0, 16000.0, 44100, kind=kind)
            mags = port.Stft(1, n, hop, kind="port").process(x[:1])["mags"]
            if mags.shape[1]:
                co, mb = mf.process(mags)
                yield f"mfcc (n {n}, {nf} filters, {nc} coeffs)", co
                yield f"melbands (n {n}, {nf} filters)", mb
    reference.check(run)
