#!/usr/bin/env python
"""Regenerates the committed golden vectors from the REAL reference.

Run in the build container (needs /root/reference and oracle/_ref/libpercepnet_ref.so, i.e. the
unmodified reference sources compiled by oracle/Makefile):

    python tests/golden/make_golden.py

Writes (all small, committed):
  toy_layers.npz   the reference's own known-answer vectors, parsed from
                   /root/reference/tests/nnet_data_test.h (tests/testnnet.cpp:19-66)
  e2e.npz          int16 input (speech+noise mix of /root/reference/sampledata, 48 hops), and what the
                   compiled reference returned for it through the float C API at both amplitude
                   scales (out, g/r) and through the CLI's int16 conversions (src/main.cpp:30-39),
                   with weights = percepnet_b200.weights.synth_model(0) (digest stored)
  stages.npz       per-stage outputs of the reference's non-static functions on the same audio
  train.npz        two (speech, noisy) int16 pairs cut from /root/reference/sampledata and the 138-float records
                   the reference's own train() (src/denoise.cpp:600) wrote for them
  reference_digests.json
                   digests (tests/util.py digest) of what the reference returned for every input of
                   tests/test_oracle_vs_reference.py, the arrays its exporter dump_percepnet.py emits for
                   synth_state_dict(3) (tests/test_weights_layout.py) and its CLI's output for e2e.npz's input;
                   the tansig table of src/tansig_table.h and the cases of the two property tests
  cli.npz          the reference CLI's PCM output and feature_test.raw for 60 synthetic hops (tests/test_dropin_cli.py)

    python tests/golden/make_golden.py --reference-digests      # the last two only
"""
import json
import os
import pathlib
import re
import subprocess
import sys
import tempfile
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle.ffi import Reference, build  # noqa: E402
from percepnet_b200.weights import synth_model  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"


def parse_arrays(path):
    txt = open(path).read()
    arrs = {}
    for m in re.finditer(r"static const float (\w+)\[(\d+)\] = \{([^}]*)\}", txt):
        arrs[m.group(1)] = np.array([float(v) for v in m.group(3).replace("\n", " ").split(",") if v.strip()],
                                    dtype=np.float32)
        assert arrs[m.group(1)].size == int(m.group(2))
    return arrs


def make_train(R):
    import tempfile
    n = 40
    sp = np.fromfile(os.path.join(REF, "sampledata/speech/speech.pcm"), dtype=np.int16)
    no = np.fromfile(os.path.join(REF, "sampledata/noise/noise.pcm"), dtype=np.int16)
    speech, noisy, recs = [], [], []
    with tempfile.TemporaryDirectory() as d:
        for k, (off, shift) in enumerate(((480 * 100, 1), (480 * 260, 3))):
            c = sp[off:off + 480 * n].copy()
            y = np.clip(c.astype(np.int32) + (no[off:off + 480 * n].astype(np.int32) >> shift), -32768, 32767).astype(np.int16)
            fc, fn, fo = (os.path.join(d, f"{nm}{k}") for nm in ("c", "n", "o"))
            c.tofile(fc); y.tofile(fn)
            assert R.train_files(fc, fn, n, fo) == 0
            speech.append(c); noisy.append(y)
            recs.append(np.fromfile(fo, np.float32).reshape(n, 138))
    np.savez_compressed(os.path.join(OUT, "train.npz"), speech=np.stack(speech), noisy=np.stack(noisy),
                        records=np.stack(recs))
    print("train.npz", os.path.getsize(os.path.join(OUT, "train.npz")))


class RefAsOracle:
    """The compiled reference behind the oracle's interface, for the *_outputs functions of
    tests/test_oracle_vs_reference.py.  The stage functions share their signatures; the reference takes its model
    through set_model."""

    def __init__(self, R):
        self.R = R

    def __getattr__(self, name):
        return getattr(self.R, name)

    def pitch_search(self, lp):
        # the reference returns no coarse correlation: it is pitch_xcorr of the decimated buffers (src/pitch.cpp)
        p, c = self.R.pitch_search(lp)
        return p, c, self.R.pitch_xcorr(lp[384::2][:240].copy(), lp[::2][:387].copy(), 147), None

    def compute_rnn(self, model, state, features):
        self.R.set_model(model)
        return self.R.compute_rnn(state, features)

    def create(self, model):
        self.R.set_model(model)
        return self.R.create()

    def process_stream(self, h, x, want_gr=False):
        out, gr = self.R.process_stream(h, x, want_gr)
        return out, gr, None

    def run_pcm16(self, model, pcm16):
        self.R.set_model(model)
        return self.R.run_pcm16(pcm16)

    def process_streams(self, model, x, n_threads=1):
        self.R.set_model(model)
        return self.R.process_streams(x, n_threads)


def property_cases():
    """The fixed cases of the two property tests: every corner of the parameter box the tests describe, then
    uniform draws."""
    rng = np.random.RandomState(2718)
    sig = [dict(seed=0, log_amp=-4.0, f0=55.0, noise=0.0, dc=-0.2, gap=0, click=False),
           dict(seed=2 ** 31 - 1, log_amp=4.5, f0=900.0, noise=1.0, dc=0.2, gap=8, click=True),
           dict(seed=1, log_amp=0.0, f0=55.0, noise=0.0, dc=0.0, gap=8, click=False),
           dict(seed=2, log_amp=4.5, f0=900.0, noise=0.0, dc=0.0, gap=0, click=True)]
    while len(sig) < 30:
        sig.append(dict(seed=int(rng.randint(0, 2 ** 31 - 1)), log_amp=float(rng.uniform(-4.0, 4.5)),
                        f0=float(rng.uniform(55.0, 900.0)), noise=float(rng.rand()), dc=float(rng.uniform(-0.2, 0.2)),
                        gap=int(rng.randint(0, 9)), click=bool(rng.rand() < 0.5)))
    pairs = [dict(seed=0, f0=60.0, snr_db=-10.0, log_level=-3.5, gap_c=0, gap_n=0),
             dict(seed=2 ** 31 - 1, f0=700.0, snr_db=40.0, log_level=0.3, gap_c=6, gap_n=6),
             dict(seed=1, f0=60.0, snr_db=40.0, log_level=0.3, gap_c=6, gap_n=0)]
    while len(pairs) < 20:
        pairs.append(dict(seed=int(rng.randint(0, 2 ** 31 - 1)), f0=float(rng.uniform(60.0, 700.0)),
                          snr_db=float(rng.uniform(-10.0, 40.0)), log_level=float(rng.uniform(-3.5, 0.3)),
                          gap_c=int(rng.randint(0, 7)), gap_n=int(rng.randint(0, 7))))
    return sig, pairs


def exporter_arrays():
    """Runs the reference's exporter (dump_percepnet.py, its dump_data methods) on its own PercepNet module loaded
    with synth_state_dict(3) -> (state_dict shapes, layer names, {array name: float32 array})."""
    import torch
    from percepnet_b200.weights import synth_state_dict
    for m in ("h5py", "tensorboardX", "matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(m, types.ModuleType(m))
    sys.modules["tensorboardX"].SummaryWriter = object
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["matplotlib.pyplot"].switch_backend = lambda *a, **k: None
    sys.path.insert(0, REF)
    import io
    import dump_percepnet  # noqa: F401  (patches Linear/Conv1d/GRU/Sequential with dump_data)
    import rnn_train
    sd = synth_state_dict(3)
    net = rnn_train.PercepNet()
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    arrays = {}
    for name, module in net.named_children():
        if name in ("gru2", "gru3", "gru_gb", "conv2"):       # the big 512x512 GRUs share code with gru_rb
            continue
        f = io.StringIO()
        module.dump_data(f, name)
        for m in re.finditer(r"static const float (\w+)\[(\d+)\] = \{([^}]*)\}", f.getvalue()):
            arrays[m.group(1)] = np.array([np.float32(v) for v in m.group(3).replace("\n", " ").split(",") if v.strip()],
                                          dtype=np.float32)
            assert arrays[m.group(1)].size == int(m.group(2))
    shapes = {k: list(v.shape) for k, v in net.state_dict().items()}
    return shapes, [n for n, _ in net.named_children()], arrays


def run_ref_cli(pcm16):
    """The reference's CLI (src/main.cpp with the exporter's nnet_data.cpp for synth_state_dict(0), oracle/Makefile)
    on int16 PCM -> (output PCM, feature_test.raw as [hops, 68])."""
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "-s", "_ref/percepNet_run_ref"], check=True)
    with tempfile.TemporaryDirectory() as d:
        pcm16.tofile(os.path.join(d, "in.pcm"))
        subprocess.run([os.path.join(ROOT, "oracle", "_ref", "percepNet_run_ref"), "in.pcm", "out.pcm"], cwd=d,
                       check=True, timeout=300)
        return (np.fromfile(os.path.join(d, "out.pcm"), dtype=np.int16),
                np.fromfile(os.path.join(d, "feature_test.raw"), dtype=np.float32).reshape(-1, 68))


def make_reference_digests(R):
    import test_oracle_vs_reference as T
    from percepnet_b200.synth import synth_pcm, to_int16
    from util import REFERENCE_DIGESTS, digest

    def digests(outputs):
        d = {}
        for key, a in outputs:
            assert d.setdefault(key, digest(a)) == digest(a), key
        return d

    impl, m0, m_hot = RefAsOracle(R), synth_model(0), synth_model(7, gain=3.0)
    sig_cases, pair_cases = property_cases()
    tmp = tempfile.TemporaryDirectory()
    tmp_path = pathlib.Path(tmp.name)

    def records(fc, fn, count):
        fo = str(tmp_path / "o")
        assert R.train_files(fc, fn, count, fo) == 0
        return np.fromfile(fo, np.float32).reshape(count, 138)

    txt = open(os.path.join(REF, "src/tansig_table.h")).read()
    res = {
        "tansig_table": [float(np.float32(v)) for v in re.findall(r"([0-9]\.[0-9]+)f", txt)],
        "erb_borders": digests(T.erb_borders_outputs(impl)),
        "fft960": digests(T.fft960_outputs(impl, np.random.RandomState(1234))),
        "band_ops": digests(T.band_ops_outputs(impl, np.random.RandomState(1234))),
        "pitch_chain": digests(T.pitch_chain_outputs(impl, np.random.RandomState(1234))),
        "network_layers": digests(T.network_layers_outputs(impl, (m0, m_hot), np.random.RandomState(1234))),
        "hot_weights": digests(T.hot_weights_outputs(impl, m_hot)),
        "multi_stream": digests(T.multi_stream_outputs(impl, m0)),
        "training_records": digests(T.training_records_outputs(records, tmp_path)),
        "training_wraparound": digests(T.training_wraparound_outputs(records, tmp_path)),
        "random_signals_cases": sig_cases,
        "random_signals": digests(T.random_signals_outputs(impl, m0, sig_cases)),
        "random_pairs_cases": pair_cases,
        "random_pairs": digests(T.random_pairs_outputs(records, pair_cases, tmp_path)),
    }
    for scale in (1.0, 32768.0):
        res[f"edge_signals/{scale:g}"] = digests(T.edge_signals_outputs(impl, m0, scale))
    tmp.cleanup()
    shapes, layers, arrays = exporter_arrays()
    res["exporter"] = {"state_dict_shapes": shapes, "layers": layers, "arrays": {k: digest(v) for k, v in arrays.items()}}
    e2e = np.load(os.path.join(OUT, "e2e.npz"))
    out16, gr = run_ref_cli(e2e["x16"])
    res["cli"] = {"e2e_out16": digest(out16), "e2e_gr": digest(gr)}
    with open(REFERENCE_DIGESTS, "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
        f.write("\n")
    out16, gr = run_ref_cli(to_int16(synth_pcm(1, 60, seed=2024)[0]))
    np.savez_compressed(os.path.join(OUT, "cli.npz"), out16=out16, gr=gr)
    for f in (REFERENCE_DIGESTS, os.path.join(OUT, "cli.npz")):
        print(os.path.basename(f), os.path.getsize(f))


def main():
    build()
    if "--train-only" in sys.argv:
        return make_train(Reference())
    if "--reference-digests" in sys.argv:
        return make_reference_digests(Reference())
    R = Reference()
    np.savez_compressed(os.path.join(OUT, "toy_layers.npz"), **parse_arrays(os.path.join(REF, "tests/nnet_data_test.h")))

    m = synth_model(0)
    R.set_model(m)
    n = 48
    sp = np.fromfile(os.path.join(REF, "sampledata/speech/speech.pcm"), dtype=np.int16)
    no = np.fromfile(os.path.join(REF, "sampledata/noise/noise.pcm"), dtype=np.int16)
    off = 480 * 100
    x16 = (sp[off:off + 480 * n].astype(np.int32) // 2 + no[off:off + 480 * n].astype(np.int32) // 2).astype(np.int16)
    res = {"x16": x16, "digest": np.frombuffer(m.digest().encode(), dtype=np.uint8)}
    for name, scale in (("unit", np.float32(1.0 / 32768.0)), ("int16", np.float32(1.0))):
        x = x16.astype(np.float32) * scale
        h = R.create()
        out, gr = R.process_stream(h, x, True)
        R.destroy(h)
        res[f"out_{name}"] = out
        res[f"gr_{name}"] = gr
    o16, gr16 = R.run_pcm16(x16)
    res["cli_out16"] = o16
    res["cli_gr"] = gr16
    np.savez_compressed(os.path.join(OUT, "e2e.npz"), **res)

    # stage taps from reference functions
    st = {}
    x = x16.astype(np.float32)
    bufs = np.stack([x[480 * k:480 * k + 1728] for k in (3, 9, 17, 30)])
    st["pitch_buf"] = bufs
    lps, ps, cs, ts, gs = [], [], [], [], []
    prev_p, prev_g = 0, 0.0
    for b in bufs:
        lp = R.pitch_downsample(b)
        p, c = R.pitch_search(lp)
        T, g = R.remove_doubling(lp, 768 - p, prev_p, prev_g)
        prev_p, prev_g = T, g
        lps.append(lp); ps.append(p); cs.append(c); ts.append(T); gs.append(g)
    st["lp"] = np.stack(lps)
    st["pitch"] = np.array(ps, np.int32)
    st["corr"] = np.array(cs, np.float32)
    st["T"] = np.array(ts, np.int32)
    st["gain"] = np.array(gs, np.float32)
    rng = np.random.RandomState(5)
    z = rng.randn(1920).astype(np.float32)
    st["fft_in"] = z
    st["fft_out"] = R.fft960(z)
    X = st["fft_out"][:962]
    P = R.fft960(rng.randn(1920).astype(np.float32))[:962]
    st["P"] = P
    st["band_energy"] = R.band_energy(X)
    st["band_corr"] = R.band_corr(X, P)
    gb = rng.rand(34).astype(np.float32)
    st["gains"] = gb
    st["interp"] = R.interp_band_gain(gb)
    st["pitch_filter"] = R.pitch_filter(X, P, gb)
    feat = (rng.rand(70) * 3).astype(np.float32)
    state = np.zeros(512 + 1024 + 4 * 512 + 128, np.float32)
    outs = []
    for _ in range(3):
        g, r = R.compute_rnn(state, feat)
        outs.append(np.concatenate([g, r]))
    st["rnn_feat"] = feat
    st["rnn_out"] = np.stack(outs)
    st["borders"] = R.erb_borders()
    np.savez_compressed(os.path.join(OUT, "stages.npz"), **st)
    make_train(R)
    for f in ("toy_layers.npz", "e2e.npz", "stages.npz"):
        print(f, os.path.getsize(os.path.join(OUT, f)))
    make_reference_digests(R)


if __name__ == "__main__":
    main()
