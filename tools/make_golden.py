"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported from /root/reference with the stub
recipe of oracle/ref_import.py) on seeded synthetic checkpoints.  Only runs in the build container.

    python tools/make_golden.py
The fixtures pin (a) the oracle restatements on any machine (tests/test_golden_cpu.py) and (b) the CUDA path on
the GPU box (tests/test_golden_gpu.py), where /root/reference does not exist.
"""
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from aicovergen_b200.synthetic import (make_hubert_state_dict, make_mdx_state_dict, make_rmvpe_state_dict,  # noqa: E402
                                       make_rvc_checkpoint)
from oracle import hubert as ohub  # noqa: E402
from oracle import mdx as om  # noqa: E402
from oracle import ref_import  # noqa: E402
from refshim import HubertShim, ref_net_g, ref_rmvpe, ref_vc  # noqa: E402
from siggen import stereo_tones, vocal_like  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)


def synth():
    cpt = make_rvc_checkpoint("40k", "v2", seed=1234)
    net = ref_net_g(cpt)
    P = 40
    g = torch.Generator().manual_seed(21)
    phone = torch.randn(1, P, 768, generator=g)
    pitch = torch.randint(1, 255, (1, P), generator=g)
    pitchf = (180 + 60 * torch.sin(torch.arange(P) * 0.2))[None].float()
    pitchf[:, 11:17] = 0
    torch.manual_seed(77)
    with torch.no_grad():
        o, _, (z, z_p, m_p, logs_p) = net.infer(phone, torch.tensor([P]), pitch, pitchf, torch.tensor([0]))
    np.savez_compressed(os.path.join(OUT, "synth_v2_40k.npz"), phone=phone.numpy(), pitch=pitch.numpy(), pitchf=pitchf.numpy(),
                        noise_seed=77, ckpt_seed=1234, out=o.numpy()[0, 0], m_p=m_p.numpy(), z=z.numpy())


def rmvpe():
    sd = make_rmvpe_state_dict(seed=4321)
    rm = ref_rmvpe(sd)
    x = vocal_like(1.6, seed=11)
    f0 = rm.infer_from_audio(x, 0.03)
    with torch.no_grad():
        hid = rm.mel2hidden(rm.mel_extractor(torch.from_numpy(x)[None]))[0].numpy()
    np.savez_compressed(os.path.join(OUT, "rmvpe.npz"), seconds=1.6, audio_seed=11, f0=f0, salience_argmax=hid.argmax(1), ckpt_seed=4321,
                        salience_max=hid.max(1))


def pipeline():
    hsd, rsd, cpt = make_hubert_state_dict(seed=777), make_rmvpe_state_dict(seed=4321), make_rvc_checkpoint("40k", "v2", seed=1234)
    audio = vocal_like(3.4, seed=13)
    xs = dict(x_pad=1, x_query=1, x_center=1, x_max=2)
    _, vc = ref_vc(40000, **xs)
    vc.model_rmvpe = ref_rmvpe(rsd)
    net = ref_net_g(cpt)
    torch.manual_seed(9)
    out = vc.pipeline(HubertShim(hsd), net, 0, audio.copy(), "x.wav", [0, 0, 0], 0, "rmvpe", "", 0.5, 1, 3, 40000, 0, 0.25,
                      "v2", 0.33, 128)
    np.savez_compressed(os.path.join(OUT, "vc_pipeline.npz"), seconds=3.4, audio_seed=13, out_int16=out, noise_seed=9, **{k: np.int64(v) for k, v in xs.items()})


def mdx():
    ref = ref_import.module("mdx")
    dim_f, dim_t, n_fft = 256, 16, 2048
    sd = make_mdx_state_dict(dim_f=dim_f, dim_t=dim_t, g=8, n=3, seed=2024)

    class FakeSession:
        def __init__(self, path, providers=None):
            pass

        def run(self, _, feed):
            return [om.convtdfnet(sd, torch.from_numpy(feed["input"])).numpy()]

    sys.modules["onnxruntime"].InferenceSession = FakeSession
    ref.ort.InferenceSession = FakeSession
    model = ref.MDXModel(torch.device("cpu"), dim_f=dim_f, dim_t=dim_t, n_fft=n_fft, stem_name="Vocals", compensation=1.035)
    sess = ref.MDX("fake.onnx", model, processor=-1)
    n = 44100 * 2 + 4321        # > 2 margins so both halves keep something
    wave = stereo_tones(n, seed=4)
    out = sess.process_wave(wave.copy(), 2)
    spec = model.stft(torch.from_numpy(wave[:, :model.chunk_size].copy())[None])
    np.savez_compressed(os.path.join(OUT, "mdx_small.npz"), n=n, wave_seed=4, processed=out.astype(np.float32), dim_f=dim_f, dim_t=dim_t,
                        n_fft=n_fft, ckpt_seed=2024, stft_abs_sum=float(spec.abs().sum()), spec_slice=spec[0, :, :8, :4].numpy())


def windows(n, count=4, width=2048):
    """Start offsets of `count` evenly spaced windows of `width` samples covering both ends of an n-sample signal."""
    return np.linspace(0, n - width, count).astype(np.int64)


def reference_pins():
    """What tests/test_oracle_vs_reference.py compares the oracle restatements against: the reference's own outputs on the
    inputs that test regenerates, plus the parameter names and shapes its model classes declare.  Long outputs are kept as
    fixed windows (windows() above) or strided samples so that the fixture stays small."""
    from aicovergen_b200.synthetic import make_ivf_index_data
    from oracle.index import IvfFlatIndex

    pins = {}
    # synthesizer: SynthesizerTrnMs768NSFsid.infer with the global CPU generator seeded (as the pipeline does)
    cpt = make_rvc_checkpoint("40k", "v2")
    net = ref_net_g(cpt)
    P = 48
    g = torch.Generator().manual_seed(1)
    phone = torch.randn(1, P, 768, generator=g)
    pitch = torch.randint(1, 255, (1, P), generator=g)
    pitchf = torch.rand(1, P, generator=g) * 300 + 80
    pitchf[:, 7:15] = 0
    torch.manual_seed(11)
    with torch.no_grad():
        o = net.infer(phone, torch.tensor([P]), pitch, pitchf, torch.tensor([0]))[0].numpy()[0, 0]
    pins["synth_starts"] = windows(len(o))
    pins["synth_out"] = np.stack([o[s:s + 2048] for s in pins["synth_starts"]])

    # rmvpe: infer_from_audio, the log-mel front end, and decode on the reference's own salience
    sd = make_rmvpe_state_dict()
    rm = ref_rmvpe(sd)
    x = vocal_like(2.5)
    pins["rmvpe_f0"] = rm.infer_from_audio(x, 0.03)
    with torch.no_grad():
        mel = rm.mel_extractor(torch.from_numpy(x)[None])
        hid = rm.mel2hidden(mel)[0].numpy()
    pins["rmvpe_mel"] = mel[0, :, ::4].numpy()                 # every 4th frame
    pins["rmvpe_salience"] = hid[::16].copy()                  # every 16th frame
    pins["rmvpe_salience_f0"] = rm.decode(pins["rmvpe_salience"].copy(), 0.03)

    # VC.pipeline with a 2-layer HuBERT, 2 segments, with and without an index (faiss.read_index returns the oracle's)
    hsd = make_hubert_state_dict(layers=2)
    audio = vocal_like(5.3)
    xs = dict(x_pad=1, x_query=1, x_center=2, x_max=3)
    base = ohub.extract_features(hsd, torch.from_numpy(vocal_like(3.0, seed=3))[None], 2)[0]
    index = IvfFlatIndex(*make_ivf_index_data(base, n_total=2000, nlist=40))

    class Shim(HubertShim):
        def extract_features(self, source, padding_mask, output_layer):
            return (ohub.extract_features(self.sd, source.float(), 2), padding_mask)

    sys.modules["faiss"].read_index = lambda p: index
    with tempfile.NamedTemporaryFile(suffix=".index") as tmp:      # the reference only reads an index file that exists
        for with_index in (False, True):
            _, vc = ref_vc(40000, **xs)
            vc.model_rmvpe = ref_rmvpe(sd)
            net_g = ref_net_g(cpt)      # built before seeding: module construction consumes RNG draws
            torch.manual_seed(5)
            out = vc.pipeline(Shim(hsd), net_g, 0, audio.copy(), "x.wav", [0, 0, 0], 0, "rmvpe", tmp.name if with_index else "",
                              0.5, 1, 3, 40000, 0, 0.25, "v2", 0.33, 128)
            pins[f"pipeline_len_{int(with_index)}"] = np.int64(len(out))
            pins[f"pipeline_starts_{int(with_index)}"] = windows(len(out))
            pins[f"pipeline_out_{int(with_index)}"] = np.stack([out[s:s + 2048] for s in windows(len(out))])

    # mdx: MDXModel.stft / istft on one chunk and MDX.process_wave (2 threads) with a session running the restated net
    ref = ref_import.module("mdx")
    dim_f, dim_t, n_fft = 256, 16, 2048
    msd = make_mdx_state_dict(dim_f=dim_f, dim_t=dim_t, g=8, n=3)

    class FakeSession:
        def __init__(self, path, providers=None):
            pass

        def run(self, _, feed):
            return [om.convtdfnet(msd, torch.from_numpy(feed["input"])).numpy()]

    sys.modules["onnxruntime"].InferenceSession = FakeSession
    ref.ort.InferenceSession = FakeSession
    model = ref.MDXModel(torch.device("cpu"), dim_f=dim_f, dim_t=dim_t, n_fft=n_fft, stem_name="Vocals", compensation=1.035)
    sess = ref.MDX("fake.onnx", model, processor=-1)
    rng = np.random.default_rng(0)
    wave = (rng.standard_normal((2, 44100 * 3 + 1234)) * 0.2).astype(np.float32)
    spec = model.stft(torch.from_numpy(wave[:, :model.chunk_size].copy())[None])
    pins["mdx_spec"] = spec[0, :, ::4].numpy()                 # every 4th frequency bin
    chunk = model.istft(spec)[0].numpy()
    pins["mdx_istft_starts"] = windows(chunk.shape[-1], width=1024)
    pins["mdx_istft"] = np.stack([chunk[:, s:s + 1024] for s in pins["mdx_istft_starts"]])
    processed = sess.process_wave(wave.copy(), 2)
    pins["mdx_len"] = np.int64(processed.shape[-1])
    pins["mdx_starts"] = windows(processed.shape[-1], width=1024)
    pins["mdx_processed"] = np.stack([processed[:, s:s + 1024] for s in pins["mdx_starts"]])

    # parameter names and shapes of the reference's model classes (what a strict load_state_dict checks), one
    # "name dim0xdim1..." line per entry
    manifest = lambda module: np.array("\n".join(f"{k} {'x'.join(map(str, v.shape))}" for k, v in sorted(module.state_dict().items())))
    m = ref_import.module("infer_pack.models")
    for key in ("40k", "48k_v2", "32k"):
        net = m.SynthesizerTrnMs768NSFsid(*make_rvc_checkpoint(key, "v2")["config"], is_half=False)
        del net.enc_q
        pins[f"state_dict_synth_{key}"] = manifest(net)
    pins["state_dict_rmvpe"] = manifest(ref_import.module("rmvpe").E2E(4, 1, (2, 2)))
    np.savez_compressed(os.path.join(OUT, "oracle_vs_reference.npz"), **pins)


if __name__ == "__main__":
    # python tools/make_golden.py [synth rmvpe pipeline mdx reference_pins]   (default: all)
    for name in sys.argv[1:] or ("synth", "rmvpe", "pipeline", "mdx", "reference_pins"):
        globals()[name]()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
