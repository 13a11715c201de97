"""Voice patches (include/maxib200.h mxb_patch; tests/patch_cases.py) on the CPU: the plain-C interpreter of oracle/maxi_oracle.c
against the same stage lists run by the reference's own objects (oracle/ref_shim.cpp) -- bit for bit, outputs, buses and the state
of every stage (live where the compiled reference is built, from its stored trace everywhere: tests/reference_trace.py) -- and
against the committed fixture tests/golden/patches.npz."""
import numpy as np
import pytest

import golden_checks as G
import patch_cases as PC

SLOTS = {1: 2, 2: 4, 3: 4, 4: 12, 5: 2, 6: 3, 7: 2, 8: 2, 10: 1, 11: 3}      # state slots per op (include/maxib200.h)


def _tables(port):
    g = G.load("tables")
    port.set_tables(g["sine"], g["transition"], float(g["sine_before"]), "port")
    return g


def test_tables_fixture_is_the_references(port, reference):
    g = G.load("tables")
    assert g["sine"].size == 514 and g["transition"].size == 1001

    def run(kind):
        s, t, b = (g["sine"], g["transition"], float(g["sine_before"])) if kind == "port" else port.get_tables("reference")
        yield "sine", s
        yield "transition", t
        yield "sine_before", b
    reference.check(run)


@pytest.mark.parametrize("case", PC.cases(), ids=lambda c: c[0])
def test_patch_port_equals_reference(port, reference, case):
    name, d, params, inputs, exact, taps = case
    _tables(port)

    def run(kind):
        V, B = 24, 200
        pa = port.Patch(d, V, delay_taps=taps, kind=kind)
        for k, v in params(V, 11).items():
            pa.set(k, v)
        for blk in range(3):
            o, m = pa.process(B, inputs(V, B, blk, 7), want_mix=True)
            assert np.isfinite(o).all() and np.abs(o).max() > 1e-3
            yield f"out {blk}", o
            yield f"mix {blk}", m
        for si, (op, kd, dst, src) in enumerate(d.stages):
            for sl in range(SLOTS.get(op, 0)):
                if op == 5 and kd in (5, 6) and sl == 1:
                    continue                                   # lopass / hipass keep one value (outputs[0])
                if op == 4 and sl == 3:
                    continue                                   # nxcHappened is indeterminate in the reference until the first trigger
                yield f"stage {si} slot {sl}", pa.get_state(si, sl)
            if op in (10, 11):
                for v in range(0, V, 5):
                    yield f"stage {si} ring {v}", pa.ring(si, v, taps)
    reference.check(run)


@pytest.mark.parametrize("case", PC.cases(), ids=lambda c: c[0])
def test_patch_golden_exact(port, case):
    """tests/golden/patches.npz (made by the compiled reference) replayed through the C port: exact, wherever gcc runs."""
    name, d, params, inputs, exact, taps = case
    _tables(port)
    g = G.load("patches")
    V, B, NB = int(g["V"]), int(g["B"]), int(g["NB"])
    p = port.Patch(d, V, delay_taps=taps, kind="port")
    for k, v in params(V, 2468).items():
        p.set(k, v)
    for blk in range(NB):
        ins = {k: g[f"{name}/in/{k}/{blk}"] for k in d.inputs}
        o, m = p.process(B, ins, want_mix=True)
        assert np.array_equal(o, g[name + "/out"][blk], equal_nan=True), (name, blk)
        assert np.array_equal(m, g[name + "/mix"][blk], equal_nan=True), (name, blk)


def test_chorus_port_equals_reference(port, reference):
    """maxiChorus: the reference draws its noise from libc rand(); the port is fed the sequence the same libc produces after the same
    srand (oracle_py.noise_fill), in the (frame, voice) order the reference's loop draws it. Outputs, buses, both delay lines' indices
    and contents, the lores state: bit for bit."""
    name, d, params, _, exact, taps = PC.chorus()
    V, B, NB, seed = 9, 150, 3, 777
    noise = port.noise_fill(seed, NB * B * V, "port").reshape(NB, B, V)
    assert np.abs(noise).max() <= 1.0 and noise.std() > 0.5
    si = [i for i, st in enumerate(d.stages) if st[0] == 18][0]

    def run(kind):
        yield "noise", noise if kind == "port" else port.noise_fill(seed, NB * B * V, kind).reshape(NB, B, V)
        pa = port.Patch(d, V, delay_taps=taps, kind=kind)
        for k, v in params(V, 3).items():
            pa.set(k, v)
        if kind == "reference":
            port.srand(seed, kind)
        for blk in range(NB):
            o, m = pa.process(B, {"noise": noise[blk]}, want_mix=True)     # the reference draws from rand() itself
            assert np.isfinite(o).all() and np.abs(o).max() > 1e-3
            yield f"out {blk}", o
            yield f"mix {blk}", m
        for sl in range(4):
            yield f"slot {sl}", pa.get_state(si, sl)
        for v in range(V):
            yield f"ring {v}", pa.ring(si, v, 2 * taps)
        if kind == "port":      # the lines are swept: indices diverged
            assert len({int(x) for x in pa.get_state(si, 0)} | {int(x) for x in pa.get_state(si, 1)}) > 2
    reference.check(run)


def test_chorus_golden_exact(port):
    g = G.load("chorus")
    name, d, params, _, exact, taps = PC.chorus()
    V, B, NB = int(g["V"]), int(g["B"]), int(g["NB"])
    assert int(g["taps"]) == taps
    p = port.Patch(d, V, delay_taps=taps, kind="port")
    for k, v in params(V, 99).items():
        p.set(k, v)
    for blk in range(NB):
        o, m = p.process(B, {"noise": g["noise"][blk]}, want_mix=True)
        assert np.array_equal(o, g["out"][blk]) and np.array_equal(m, g["mix"][blk]), blk


def test_registers_read_zero_until_written(port):
    from maximilian_b200.patchdef import PatchDef, R
    d = PatchDef()
    d.stage("add", R(3), d.K(1.5), dst=R(0))        # R3 was written by the PREVIOUS sample's last stage: must read 0 here
    d.stage("out", R(0))
    d.stage("add", R(0), d.K(1.0), dst=R(3))
    o, _ = port.Patch(d, 3, kind="port").process(4)
    assert np.all(o == 1.5)
