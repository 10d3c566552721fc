"""Pins the oracle restatements against the UNMODIFIED reference code.  What the reference computed on the inputs below, and
the parameter names and shapes its model classes declare, were recorded by tools/make_golden.py into
tests/golden/oracle_vs_reference.npz (long outputs as fixed windows or strided samples).  Where the two used to be compared
bit for bit within one process they are held to a few float32 ulps here: the recording was made on another CPU, whose BLAS and
FFT may sum in another order (the rmvpe log-mel already moves by half an ulp between 1 and 8 threads on one machine)."""
import os

import numpy as np
import pytest
import torch

from siggen import vocal_like

PINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_reference.npz")
ULPS = 8


def ulps(got, want):
    """Largest |got - want| in float32 ulps of the largest |want|."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    return float(np.abs(got - want).max() / (np.finfo(np.float32).eps * np.abs(want).max()))


def windows(x, starts, width):
    return np.stack([x[..., s:s + width] for s in starts])


def test_synth_oracle_matches_reference():
    from aicovergen_b200.synthetic import make_rvc_checkpoint
    from oracle import synth as osyn

    z = np.load(PINS)
    cpt = make_rvc_checkpoint("40k", "v2")
    P = 48
    g = torch.Generator().manual_seed(1)
    phone = torch.randn(1, P, 768, generator=g)
    pitch = torch.randint(1, 255, (1, P), generator=g)
    pitchf = torch.rand(1, P, generator=g) * 300 + 80
    pitchf[:, 7:15] = 0
    nz, ns = osyn.draw_noise(11, P, 192, 400)
    o = osyn.infer(cpt, phone, pitch, pitchf, torch.tensor([0]), nz, ns).numpy()[0, 0]
    assert o.shape == (z["synth_starts"][-1] + 2048,)
    assert np.abs(windows(o, z["synth_starts"], 2048) - z["synth_out"]).max() < 2e-6


def test_synthetic_checkpoints_load_strictly_in_reference():
    """The synthetic checkpoints carry exactly the parameter names and shapes of the reference's model classes (what
    load_state_dict checks: no missing or unexpected key, no size mismatch)."""
    from aicovergen_b200.synthetic import make_rmvpe_state_dict, make_rvc_checkpoint

    z = np.load(PINS)

    def assert_loads_strictly(sd, name):
        want = dict(line.rsplit(" ", 1) for line in str(z[name]).split("\n"))
        have = {k: "x".join(map(str, v.shape)) for k, v in sd.items()}
        missing, unexpected = sorted(want.keys() - have.keys()), sorted(have.keys() - want.keys())
        wrong = sorted(k for k in want.keys() & have.keys() if want[k] != have[k])
        assert not missing and not unexpected and not wrong, (name, missing[:5], unexpected[:5], wrong[:5])

    for key, up in (("40k", 400), ("48k_v2", 480), ("32k", 320)):
        cpt = make_rvc_checkpoint(key, "v2")
        assert_loads_strictly(cpt["weight"], f"state_dict_synth_{key}")
        assert int(np.prod(cpt["config"][12])) == up
    assert_loads_strictly(make_rmvpe_state_dict(), "state_dict_rmvpe")


def test_rmvpe_oracle_matches_reference():
    from aicovergen_b200.synthetic import make_rmvpe_state_dict
    from oracle import rmvpe as orm

    z = np.load(PINS)
    sd = make_rmvpe_state_dict()
    x = vocal_like(2.5)
    f_ref = z["rmvpe_f0"]
    f_or = orm.infer_from_audio(sd, x, 0.03)
    assert f_ref.shape == f_or.shape
    assert np.abs(f_ref - f_or).max() / f_ref.max() < 1e-5
    mel = orm.log_mel(torch.from_numpy(x)[None])
    assert mel.shape == (1, 128, len(f_ref))
    assert ulps(mel[0, :, ::4].numpy(), z["rmvpe_mel"]) <= ULPS
    # decode restatement, given the reference's own salience: the same numpy operations in the same order (a CPU with
    # other vector units may round the final power differently in the last place)
    sal = z["rmvpe_salience"]
    got, want = orm.decode(sal.copy(), 0.03), z["rmvpe_salience_f0"]
    assert np.array_equal(got > 0, want > 0)
    np.testing.assert_array_max_ulp(got, want, maxulp=2)


@pytest.mark.parametrize("with_index", [False, True])
def test_pipeline_oracle_matches_reference(with_index):
    """Whole VC.pipeline: 2 segments (small x_* so it stays cheap), rmvpe F0, protect + RMS mix (+ index)."""
    from aicovergen_b200.synthetic import (make_hubert_state_dict, make_ivf_index_data, make_rmvpe_state_dict,
                                           make_rvc_checkpoint)
    from oracle import hubert as ohub
    from oracle import pipeline as opipe
    from oracle.index import IvfFlatIndex

    z = np.load(PINS)
    hsd = make_hubert_state_dict(layers=2)
    cpt = make_rvc_checkpoint("40k", "v2")
    rsd = make_rmvpe_state_dict()
    audio = vocal_like(5.3)
    xs = dict(x_pad=1, x_query=1, x_center=2, x_max=3)
    index = None
    if with_index:
        base = ohub.extract_features(hsd, torch.from_numpy(vocal_like(3.0, seed=3))[None], 2)[0]
        cent, vecs = make_ivf_index_data(base, n_total=2000, nlist=40)
        index = IvfFlatIndex(cent, vecs)
    # the reference ran with the same 2-layer hubert: temporarily patch the layer count
    orig = ohub.extract_features
    ohub.extract_features = lambda sd, src, layer=12, n_heads=12: orig(sd, src, 2, n_heads)
    try:
        out, info = opipe.pipeline(hsd, cpt, rsd, audio.copy(), index=index, seed=5, return_all=True, **xs)
    finally:
        ohub.extract_features = orig
    assert len(info["opt_ts"]) >= 1, "test must exercise the cut-point path"
    i = int(with_index)
    assert out.shape == (int(z[f"pipeline_len_{i}"]),) and out.dtype == np.int16
    diff = np.abs(windows(out, z[f"pipeline_starts_{i}"], 2048).astype(np.int32) - z[f"pipeline_out_{i}"].astype(np.int32))
    # the only arithmetic difference is fp32 reassociation in the GRU restatement (f0 differs ~1e-6 relative,
    # which the random-weight synthesizer amplifies to ~1e-4 on the waveform)
    assert diff.max() <= 12, diff.max()
    assert np.sqrt((diff.astype(np.float64) ** 2).mean()) < 1.5


def test_mdx_oracle_matches_reference():
    """mdx.py's own MDXModel.stft/istft and MDX.process_wave (2 threads, margins, padding) with a fake ORT
    session running the restated net, vs oracle/mdx.py."""
    from aicovergen_b200.synthetic import make_mdx_state_dict
    from oracle import mdx as om

    z = np.load(PINS)
    dim_f, dim_t, n_fft = 256, 16, 2048         # small geometry: chunk = 1024*15 samples, trim 1024
    sd = make_mdx_state_dict(dim_f=dim_f, dim_t=dim_t, g=8, n=3)
    net = lambda spec: om.convtdfnet(sd, spec)
    mp = om.MdxParams(dim_f, dim_t, n_fft, stem_name="Vocals", compensation=1.035)
    rng = np.random.default_rng(0)
    N = 44100 * 3 + 1234
    wave = (rng.standard_normal((2, N)) * 0.2).astype(np.float32)
    # stft / istft
    x = torch.from_numpy(wave[:, :mp.chunk_size].copy())[None]
    spec = mp.stft(x)
    assert ulps(spec[0, :, ::4].numpy(), z["mdx_spec"]) <= ULPS
    chunk = mp.istft(spec)[0].numpy()
    assert chunk.shape == (2, mp.chunk_size)
    assert ulps(windows(chunk, z["mdx_istft_starts"], 1024), z["mdx_istft"]) <= ULPS
    # full process_wave
    got = om.process_wave(wave.copy(), mp, net, 2)
    assert got.shape == wave.shape == (2, int(z["mdx_len"]))
    assert np.abs(windows(got, z["mdx_starts"], 1024) - z["mdx_processed"]).max() < 1e-6
