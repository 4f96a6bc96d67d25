"""Pins the C restatement (oracle/pn_oracle.c) to the compiled, unmodified reference, stage by stage and end to end,
BIT FOR BIT.  Every input below is rebuilt from its seed; what the reference returned for it is stored as a digest of
its bits in tests/golden/reference_digests.json, written by tests/golden/make_golden.py, which runs these same
``*_outputs`` functions on the reference.  CPU only."""
import numpy as np
import pytest

from util import digest, edge_signals, reference_digests, same_bits


def check(section, outputs):
    """Every (key, array) of `outputs` has the digest the reference's array of that key has."""
    want = reference_digests()[section]
    seen = set()
    for key, a in outputs:
        assert key in want, f"{section}: no reference output {key}"
        assert digest(a) == want[key], f"{section}: {key} differs from the reference"
        seen.add(key)
    assert seen == set(want), f"{section}: reference outputs not compared: {sorted(set(want) - seen)}"


@pytest.fixture
def rng():
    return np.random.RandomState(1234)


def erb_borders_outputs(impl):
    yield "borders", impl.erb_borders()


def test_erb_borders(oracle):
    check("erb_borders", erb_borders_outputs(oracle))
    assert oracle.erb_borders().tolist() == [0, 2, 4, 6, 8, 10, 12, 14, 16, 18, 20, 22, 24, 26, 28, 31, 36, 41, 48, 56,
                                             65, 75, 86, 99, 115, 132, 152, 175, 201, 230, 265, 304, 349, 400]   # SURVEY.md 8(a3)


def test_tansig_table_matches_header(oracle):
    """The reference's src/tansig_table.h, parsed into tests/golden/reference_digests.json."""
    vals = np.array(reference_digests()["tansig_table"], np.float32)
    assert vals.size == 201
    # tansig(0.04*i) at the table nodes returns the table value itself (x - 0.04f*i == 0 there)
    got = oracle.tansig(np.float32(0.04) * np.arange(201, dtype=np.float32))
    nodes_exact = np.float32(0.04) * np.arange(201, dtype=np.float32) - np.float32(0.04) * np.arange(201, dtype=np.float32)
    assert np.all(nodes_exact == 0)
    assert same_bits(got, vals)


def fft960_outputs(impl, rng):
    for amp in (1.0, 1e-3, 3e4):
        z = (rng.randn(1920) * amp).astype(np.float32)
        yield f"amp{amp:g}", impl.fft960(z)
    d = np.zeros(1920, np.float32); d[2 * 7] = 1
    yield "delta", impl.fft960(d)


def test_fft960(oracle, rng):
    check("fft960", fft960_outputs(oracle, rng))


def band_ops_outputs(impl, rng):
    X = (rng.randn(962) * 3).astype(np.float32)
    P = rng.randn(962).astype(np.float32)
    yield "band_energy", impl.band_energy(X)
    yield "band_corr", impl.band_corr(X, P)
    g = rng.rand(34).astype(np.float32)
    yield "interp_band_gain", impl.interp_band_gain(g)
    yield "pitch_filter", impl.pitch_filter(X, P, g)


def test_band_ops(oracle, rng):
    outs = dict(band_ops_outputs(oracle, rng))
    check("band_ops", outs.items())
    assert np.all(outs["interp_band_gain"][400:] == 0)            # SURVEY.md App. C.1


def _pitch_bufs(rng):
    t = np.arange(1728) / 48000.0
    yield (3000 * np.sin(2 * np.pi * 140 * t) + 200 * rng.randn(1728)).astype(np.float32)
    yield (0.2 * np.sin(2 * np.pi * 300 * t) + 0.01 * rng.randn(1728)).astype(np.float32)
    yield np.zeros(1728, np.float32)
    yield (rng.randn(1728) * 1e-4).astype(np.float32)
    yield (8000 * np.sign(np.sin(2 * np.pi * 62.5 * t))).astype(np.float32)
    for _ in range(6):
        f0 = rng.uniform(60, 800)
        yield (1000 * np.sin(2 * np.pi * f0 * t) + 500 * np.sin(4 * np.pi * f0 * t + 1) + 100 * rng.randn(1728)).astype(np.float32)


def pitch_chain_outputs(impl, rng):
    """Each stage on its own input: the stages after pitch_downsample all read the same decimated buffer.  The coarse
    correlation is yielded twice, from pitch_search's tap and from pitch_xcorr itself."""
    prev = (0, 0.0)
    for i, buf in enumerate(_pitch_bufs(rng)):
        lp = impl.pitch_downsample(buf)
        yield f"{i}/lp", lp
        ac, lpc = impl.autocorr_lpc(lp)
        yield f"{i}/ac", ac
        yield f"{i}/lpc", lpc
        p, c, coarse, _ = impl.pitch_search(lp)
        yield f"{i}/pitch", np.int32(p)
        yield f"{i}/corr", np.float32(c)
        yield f"{i}/coarse", coarse
        x4, y4 = lp[384::2][:240].copy(), lp[::2][:387].copy()
        yield f"{i}/coarse", impl.pitch_xcorr(x4, y4, 147)
        for k, (pp, pg) in enumerate((prev, (0, 0.0), (p // 2 * 2, 0.8), (120, 0.5))):
            T, g = impl.remove_doubling(lp, 768 - p, pp, pg)
            yield f"{i}/T{k}", np.int32(T)
            yield f"{i}/gain{k}", np.float32(g)
        prev = (T, g)


def test_pitch_chain(oracle, rng):
    check("pitch_chain", pitch_chain_outputs(oracle, rng))


def network_layers_outputs(impl, models, rng):
    for j, model in enumerate(models):
        m = model.as_c_model()
        x = (rng.rand(70) * 4).astype(np.float32)
        yield f"{j}/fc", impl.dense_layer(m.fc.contents, x, 128)
        mem = np.zeros(640, np.float32)
        for t in range(6):
            x = rng.rand(128).astype(np.float32)
            yield f"{j}/conv1/{t}", impl.conv1d_layer(m.conv1.contents, mem, x, 512)
            yield f"{j}/conv1_mem/{t}", mem.copy()
        for name, layer, M, H in (("gru1", m.gru1.contents, 512, 512), ("gru_rb", m.gru_rb.contents, 1024, 128)):
            h = np.zeros(H, np.float32)
            for t in range(4):
                x = (rng.randn(M)).astype(np.float32)
                impl.gru_layer(layer, h, x)
                yield f"{j}/{name}/{t}", h.copy()
        state = np.zeros(3712, np.float32)
        for t in range(5):
            f = (rng.rand(70) * 2).astype(np.float32)
            g, r = impl.compute_rnn(model, state, f)
            yield f"{j}/rnn_g/{t}", g
            yield f"{j}/rnn_r/{t}", r
            yield f"{j}/rnn_state/{t}", state.copy()


def test_network_layers(oracle, model0, model_hot, rng):
    check("network_layers", network_layers_outputs(oracle, (model0, model_hot), rng))


def test_activation_sweep(oracle):
    x = np.linspace(-9, 9, 4001).astype(np.float32)
    t = oracle.tansig(x)
    assert np.max(np.abs(t - np.tanh(x.astype(np.float64)))) < 2e-4   # table approximation error bound
    s = oracle.sigmoid(x)
    assert np.max(np.abs(s - 1 / (1 + np.exp(-x.astype(np.float64))))) < 1e-4


def edge_signals_outputs(impl, model, scale):
    for name, x in edge_signals(16, scale).items():
        h = impl.create(model)
        y, gr, _ = impl.process_stream(h, x, True)
        impl.destroy(h)
        yield f"{name}/out", y
        yield f"{name}/gr", gr


@pytest.mark.parametrize("scale", [1.0, 32768.0])
def test_end_to_end_edge_signals(oracle, model0, scale):
    check(f"edge_signals/{scale:g}", edge_signals_outputs(oracle, model0, scale))


def hot_weights_outputs(impl, model):
    from percepnet_b200.synth import synth_pcm, to_int16
    x16 = to_int16(synth_pcm(1, 20, seed=99)[0])
    o16, g16 = impl.run_pcm16(model, x16)
    yield "cli_out16", o16
    yield "cli_gr", g16
    x = x16.astype(np.float32)       # int16-scale floats: the comb-filter branch executes (SURVEY.md 0.6)
    h = impl.create(model)
    y, gr, _ = impl.process_stream(h, x, True)
    impl.destroy(h)
    yield "out", y
    yield "gr", gr


def test_end_to_end_hot_weights_and_cli(oracle, model_hot):
    from percepnet_b200.synth import synth_pcm, to_int16
    check("hot_weights", hot_weights_outputs(oracle, model_hot))
    x = to_int16(synth_pcm(1, 20, seed=99)[0]).astype(np.float32)
    ho = oracle.create(model_hot); _, _, taps = oracle.process_stream(ho, x, True, taps=True); oracle.destroy(ho)
    assert sum(1 for t in taps if not t.silence) >= 10


def multi_stream_outputs(impl, model):
    from percepnet_b200.synth import synth_pcm
    yield "out", impl.process_streams(model, synth_pcm(3, 6, seed=5), 2)


def test_multi_stream_driver(oracle, model0):
    check("multi_stream", multi_stream_outputs(oracle, model0))


def oracle_records(oracle):
    """The restated train() on two int16 files, read the way train() reads them (gen_features.read_cyclic_frames)."""
    from percepnet_b200.gen_features import read_cyclic_frames
    return lambda fc, fn, count: oracle.train_records(read_cyclic_frames(fc, count), read_cyclic_frames(fn, count))


def training_records_outputs(records, tmp_path):
    from percepnet_b200.synth import synth_pairs
    n_frames = 40
    clean, noisy = synth_pairs(6, n_frames, seed=77)
    cases = [(clean[k], noisy[k]) for k in range(6)]
    cases.append((np.zeros_like(clean[0]), noisy[0]))
    cases.append((noisy[1], noisy[1]))
    cases.append((clean[2], (noisy[2] // 64).astype(np.int16)))      # noisy far below clean: g clipped at 1
    for k, (c, n) in enumerate(cases):
        fc, fn = str(tmp_path / f"c{k}"), str(tmp_path / f"n{k}")
        c.tofile(fc); n.tofile(fn)
        yield str(k), records(fc, fn, n_frames)


def test_training_records_match_reference_train(oracle, tmp_path):
    """Row f1: the restated train() loop and label math (denoise.cpp:549-589, 600-787) against the reference's own
    train() run on files: every 138-float record bit for bit, over speech-like pairs at several SNRs, an
    all-zero clean file (g = 0) and identical clean/noisy files (g = 1 up to the .0001 bias)."""
    outs = list(training_records_outputs(oracle_records(oracle), tmp_path))
    check("training_records", outs)
    saw_branch = sum(int(np.any(rec[:, 104:] == np.float32(0.99))) for _, rec in outs)
    assert saw_branch >= 3        # the Ephatp < Exp branch (r = 0.99, attenuated g) is exercised


def training_wraparound_outputs(records, tmp_path):
    from percepnet_b200.synth import synth_pairs
    clean, noisy = synth_pairs(1, 12, seed=5)
    count = 30
    for tail_c, tail_n, nc, nn in ((0, 0, 12, 12), (123, 0, 9, 12), (7, 479, 12, 7)):
        fc, fn = str(tmp_path / "c"), str(tmp_path / "n")
        clean[0][:nc * 480 + tail_c].tofile(fc)
        noisy[0][:nn * 480 + tail_n].tofile(fn)
        yield f"{tail_c}/{tail_n}", records(fc, fn, count)


def test_training_file_wraparound_matches_reference(oracle, tmp_path):
    """train() re-reads a file from its start when a read hits EOF (denoise.cpp:676-679, 687-690); the CLI's
    read_cyclic_frames restates that: files shorter than <count>, with and without a trailing partial frame."""
    check("training_wraparound", training_wraparound_outputs(oracle_records(oracle), tmp_path))


def random_signal(seed, log_amp, f0, noise, dc, gap, click):
    """A mixture of a harmonic stack, noise, DC, an optional click and an optional silent gap, 14 hops."""
    n_frames = 14
    T = n_frames * 480
    rng = np.random.RandomState(seed)
    t = np.arange(T) / 48000.0
    x = np.zeros(T)
    for h in range(1, 9):
        x += rng.rand() * np.sin(2 * np.pi * f0 * h * t + rng.rand() * 6.28) / h
    x = x / (np.abs(x).max() + 1e-9) * (1 - noise) + noise * rng.randn(T) * 0.3 + dc
    if gap:
        g0 = rng.randint(0, n_frames - gap + 1) * 480
        x[g0:g0 + gap * 480] = 0.0                              # exact silence: the E < 0.1 branch
    if click:
        x[rng.randint(0, T)] += 3.0
    return (x * 10.0 ** log_amp).astype(np.float32)


def random_signals_outputs(impl, model, cases):
    for k, case in enumerate(cases):
        x = random_signal(**case)
        h = impl.create(model)
        y, gr, _ = impl.process_stream(h, x, True)
        impl.destroy(h)
        yield f"{k}/out", y
        yield f"{k}/gr", gr


def test_random_signals_end_to_end_property(oracle, model0):
    """Property test: for arbitrary mixtures of harmonic stacks, noise, DC, clicks and silent gaps at amplitudes
    from 1e-4 to full int16 scale, the restatement and the compiled reference agree bit for bit on every output
    sample and every g/r value.  The 30 cases (seed in [0, 2^31), log10 amplitude in [-4, 4.5], f0 in [55, 900] Hz,
    noise share in [0, 1], DC in [-0.2, 0.2], gap of 0-8 hops, click or not) are stored with the digests."""
    cases = reference_digests()["random_signals_cases"]
    assert len(cases) == 30
    check("random_signals", random_signals_outputs(oracle, model0, cases))


def random_pair(seed, f0, snr_db, log_level, gap_c, gap_n):
    """A (speech, noisy) int16 pair of 16 hops: a harmonic stack and the same plus noise at `snr_db`, each with an
    optional silent stretch, at 32768 * 10**log_level (clipped above full scale)."""
    n_frames = 16
    T = n_frames * 480
    rng = np.random.RandomState(seed)
    t = np.arange(T) / 48000.0
    sp = np.zeros(T)
    for h in range(1, 7):
        sp += rng.rand() * np.sin(2 * np.pi * f0 * h * t + rng.rand() * 6.28) / h
    sp /= np.abs(sp).max() + 1e-9
    noise = rng.randn(T) * 10 ** (-snr_db / 20) * 0.3
    if gap_c:
        g0 = rng.randint(0, n_frames - gap_c + 1) * 480
        sp[g0:g0 + gap_c * 480] = 0
    noisy = sp + noise
    if gap_n:
        g0 = rng.randint(0, n_frames - gap_n + 1) * 480
        noisy[g0:g0 + gap_n * 480] = 0
    lvl = 32768.0 * 10 ** log_level                                  # > 1 clips
    c16 = np.clip(np.rint(sp * lvl), -32768, 32767).astype(np.int16)
    n16 = np.clip(np.rint(noisy * lvl), -32768, 32767).astype(np.int16)
    return c16, n16


def random_pairs_outputs(records, cases, tmp_path):
    for k, case in enumerate(cases):
        c16, n16 = random_pair(**case)
        fc, fn = str(tmp_path / "c"), str(tmp_path / "n")
        c16.tofile(fc); n16.tofile(fn)
        yield str(k), records(fc, fn, 16)


def test_random_pairs_training_records_property(oracle, tmp_path):
    """Property test for row f1: random (speech, noisy) int16 pairs -- random pitch, SNR from -10 to 40 dB, random
    level down to a few LSBs, clipping, silent stretches in either file -- give bit-identical 138-float records from
    the restated loop and from the reference's own train().  The 20 cases are stored with the digests."""
    cases = reference_digests()["random_pairs_cases"]
    assert len(cases) == 20
    check("random_pairs", random_pairs_outputs(oracle_records(oracle), cases, tmp_path))
