"""Generate the committed golden fixtures from a LiveTalking checkout:

    LTB_REFERENCE=<LiveTalking checkout> python tests/golden/make_golden.py

* w2l_golden.npz   — the UNMODIFIED reference nn.Module (avatars/wav2lip/models/wav2lip_v2.py, imported by file
                     path) run on CPU fp32 with the seeded synthetic weights of oracle.wav2lip_ref.synth_state_dict(0)
                     and oracle.wav2lip_ref.synth_inputs(1, seed=5).  Pins oracle/wav2lip_ref.py to the reference code.
* paste_golden.npz — cv2.resize / LipReal.paste_back_frame semantics (avatars/wav2lip_avatar.py:141-147) produced
                     with the installed OpenCV, for several bbox sizes (up-scale, down-scale, exact 2x, identity).
* mel_golden.npz   — librosa is not installed anywhere we can reach, so the mel fixture is produced by an
                     INDEPENDENT torch pipeline (torch.stft + torchaudio Slaney filterbank + scipy.lfilter) following
                     avatars/wav2lip/audio.py:45-51; it pins oracle/mel_ref.py against a second implementation
                     ("parity unpinned" w.r.t. librosa itself, see oracle/__init__.py).
* mel_chain_golden.npz / mel_window_golden.npz — the reference's OWN audio.py + hparams.py and MelASR.run_step executed
                     here (only librosa.stft / filters.mel substituted): everything around the two librosa calls.
* slice_golden.npz — Whisper window indices from the reference's own BaseASR._get_sliced_feature.
* ultralight_golden.npz — the UNMODIFIED reference U-Net (avatars/ultralight/unet.py Model(6,'hubert'), imported by path) on
                     oracle.ultralight_ref.synth_state_dict(0) / synth_inputs(2, seed=9); LightReal.inference_batch +
                     paste_back_frame (avatars/ultralight_avatar.py:141-184) run from the reference module with that network; and
                     the window rows of the reference's own BaseASR._feature2chunks as HubertASR.run_step calls it.
* lipreal_golden.npz — LipReal.inference_batch + paste_back_frame run from the reference module (a4 + a5 + a6 glue).
* pe_golden.npz, vae_glue_golden.npz, musereal_golden.npz — the reference's PositionalEncoding, VAE.preprocess_img /
                     decode_latents and MuseReal.inference_batch (third-party networks replaced by recorders / fakes).
* asr_host_golden.npz — the reference's own BaseASR / WhisperASR / HubertASR queue bookkeeping (extractors replaced by
                     recorders) on the seeded event sequences of tests/test_plugin_host.py.
* mt_blend_golden.npz — the reference's own get_image_blending (avatars/musetalk/myutil.py) on a seeded MuseTalk paste-back.
Every generator is deterministic: re-running this script reproduces the committed files byte for byte.
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import wav2lip_ref as R  # noqa: E402

REF = os.environ.get("LTB_REFERENCE", "")


def load_reference_wav2lip():
    pk = types.ModuleType("refmodels")
    pk.__path__ = [f"{REF}/avatars/wav2lip/models"]
    sys.modules["refmodels"] = pk
    mods = {}
    for n in ("conv", "wav2lip_v2"):
        spec = importlib.util.spec_from_file_location(f"refmodels.{n}", f"{REF}/avatars/wav2lip/models/{n}.py")
        m = importlib.util.module_from_spec(spec)
        sys.modules[f"refmodels.{n}"] = m
        spec.loader.exec_module(m)
        mods[n] = m
    return mods["wav2lip_v2"].Wav2Lip


def make_w2l():
    sd = R.synth_state_dict(0)
    mel, img = R.synth_inputs(1, seed=5)
    net = load_reference_wav2lip()()
    net.load_state_dict(sd, strict=True)
    net.eval()
    taps = {}
    hooks = []
    names = [p for p, _ in R.layer_list()]
    for n in names:
        mod = net.get_submodule(n)
        hooks.append(mod.register_forward_hook(lambda m, i, o, n=n: taps.__setitem__(n, o.detach())))
    with torch.no_grad():
        out = net(mel, img)
    for h in hooks:
        h.remove()
    pred = (out.numpy().transpose(0, 2, 3, 1) * 255.0)  # wav2lip_avatar.py:138
    stats = np.array([[float(taps[n].mean()), float(taps[n].abs().mean()), float(taps[n].std())] for n in names], np.float64)
    np.savez_compressed(os.path.join(HERE, "w2l_golden.npz"),
                        pred_u8=pred.astype(np.uint8),
                        pred_f32_sub=pred[:, ::4, ::4, :].astype(np.float32),
                        layer_stats=stats,
                        audio_emb=taps["audio_encoder.12"].numpy().reshape(-1).astype(np.float32),
                        seed=np.array([0, 5]))
    print("w2l golden: pred mean", pred.mean(), "std", pred.std())


def synth_pred():
    """Deterministic (256,256,3) float prediction with fractional parts (exercises the astype(uint8) truncation)."""
    seed = np.random.default_rng(7).integers(0, 256, (32, 32, 3))
    yy, xx = np.mgrid[0:256, 0:256]
    base = np.kron(seed, np.ones((8, 8, 1), dtype=np.int64))
    u8 = (base + (xx * 3 + yy * 5)[..., None]) % 256
    return (u8 + 0.63).astype(np.float32).clip(0, 255)


def synth_frame(h, w):
    yy, xx = np.mgrid[0:h, 0:w]
    return np.stack([(yy * 2) % 256, (xx * 3) % 256, (yy + xx) % 256], -1).astype(np.uint8)


def make_paste():
    import zlib
    import cv2
    pred = synth_pred()
    # (y1,y2,x1,x2): up-scale, down-scale, exact 2x decimation (INTER_AREA substitution), identity, thin, full-frame
    boxes = np.array([[10, 110, 20, 150], [5, 69, 8, 104], [30, 31, 40, 45], [2, 118, 3, 51], [10, 138, 20, 148],
                      [20, 276, 30, 286], [0, 300, 0, 300], [7, 295, 1, 130]], np.int32)
    crcs, subs = [], []
    for (y1, y2, x1, x2) in boxes:
        comb = synth_frame(300, 300)
        comb[y1:y2, x1:x2] = cv2.resize(pred.astype(np.uint8), (int(x2 - x1), int(y2 - y1)))  # wav2lip_avatar.py:145-146
        crcs.append(zlib.crc32(comb.tobytes()))
        subs.append(comb[::3, ::3].copy())
    np.savez_compressed(os.path.join(HERE, "paste_golden.npz"), boxes=boxes, crc32=np.array(crcs, np.uint64),
                        sub=np.stack(subs))
    print("paste golden ok")


def make_mel():
    import scipy.signal
    import torchaudio
    rng = np.random.default_rng(42)
    t = np.arange(16640) / 16000.0
    pcm = (0.3 * np.sin(2 * np.pi * 440 * t) + 0.1 * np.sin(2 * np.pi * 1330 * t + 1.0) +
           0.05 * rng.standard_normal(t.size)).astype(np.float32)
    y = scipy.signal.lfilter([1, -0.97], [1], pcm)
    D = torch.stft(torch.from_numpy(y), 800, 200, 800, window=torch.hann_window(800, periodic=True, dtype=torch.float64),
                   center=True, pad_mode="constant", return_complex=True).abs().numpy()
    fb = torchaudio.functional.melscale_fbanks(401, 55.0, 7600.0, 80, 16000, norm="slaney", mel_scale="slaney").T.numpy()
    S = fb.astype(np.float64) @ D
    S = 20 * np.log10(np.maximum(1e-5, S)) - 20
    mel = np.clip(8.0 * ((S + 100.0) / 100.0) - 4.0, -4.0, 4.0)
    starts = [int(16.0 + i * 3.2) for i in range(16)]
    win = np.stack([mel[:, s:s + 16] for s in starts], 0)
    np.savez_compressed(os.path.join(HERE, "mel_golden.npz"), pcm=pcm, windows=win.astype(np.float32), mel=mel.astype(np.float32))
    print("mel golden ok", win.shape, float((win == -4).mean()))


def make_slices():
    """Window indices of the audio-feature slicing, produced by the reference's OWN code:
    BaseASR._get_sliced_feature (avatars/audio_features/base_asr.py:91-133) driven as WhisperASR._feature2chunks /
    run_step do (whisper.py:35-76: win [0,5], start = stride_left/2, multiplier 2), and the Wav2Lip mel window starts of
    MelASR.run_step (mel.py:47-63).  Pins the index arithmetic of csrc/whisper.cu::whisper_slice and csrc/mel.cu."""
    sys.path.insert(0, os.path.join(HERE, ".."))
    import stubs
    stubs.install()
    spec = importlib.util.spec_from_file_location("ref_base_asr", os.path.join(REF, "avatars/audio_features/base_asr.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    out = {}
    cfgs = [(4, 10, 1500), (16, 10, 1500), (8, 5, 1500), (32, 10, 1500), (16, 10, 40), (3, 0, 7)]   # (batch, stride_left, feature rows)
    for B, l, T in cfgs:
        asr = ref.BaseASR(stubs.Opt(batch_size=B, l=l))
        feat = np.arange(T, dtype=np.float32).reshape(T, 1)
        idx = []
        for i in range(B):                                   # WhisperASR._feature2chunks, whisper.py:48-55
            sel, sel_idx = asr._get_sliced_feature(feature_array=feat, vid_idx=i + l / 2, audio_feat_win=[0, 5], feature_idx_multiplier=2)
            assert sel.shape[0] == len(sel_idx) == 10
            idx.append(sel_idx)
        out[f"whisper_B{B}_l{l}_T{T}"] = np.asarray(idx, np.int32)
    np.savez_compressed(os.path.join(HERE, "slice_golden.npz"), cfgs=np.asarray(cfgs, np.int32), **out)
    print("slice golden ok", {k: v.shape for k, v in out.items()})


def make_pe():
    """MuseTalk audio positional encoding from the reference's OWN class (avatars/musetalk/models/unet.py:12-27), imported by
    file path with a stub standing in for the absent `diffusers` package (only the UNet wrapper below the class needs it)."""
    fake = types.ModuleType("diffusers")
    fake.UNet2DConditionModel = object
    sys.modules.setdefault("diffusers", fake)
    spec = importlib.util.spec_from_file_location("ref_mt_unet", os.path.join(REF, "avatars/musetalk/models/unet.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    pe = ref.PositionalEncoding(d_model=384)
    g = torch.Generator().manual_seed(11)
    x = torch.randn(2, 50, 384, generator=g)
    with torch.no_grad():
        y = pe(x)
    # x is regenerated from the seed by the test; keep the sinusoid table and a subsample of the module's output
    np.savez_compressed(os.path.join(HERE, "pe_golden.npz"), seed=np.int64(11), table=pe.pe[0, :50].numpy(), y_sub=y.numpy()[:, ::5, ::7])
    print("pe golden ok", tuple(y.shape))


def make_vae_glue():
    """The pre/post-processing around the (absent) diffusers VAE, executed by the reference's OWN wrapper methods
    (avatars/musetalk/models/vae.py:51-82 preprocess_img, :96-108 decode_latents) on an instance built without __init__
    (AutoencoderKL.from_pretrained needs the checkpoint) and a fake `vae` whose decode returns a fixed tensor."""
    import zlib
    fake = types.ModuleType("diffusers")
    fake.AutoencoderKL = object
    sys.modules.setdefault("diffusers", fake)
    if not hasattr(sys.modules["diffusers"], "AutoencoderKL"):
        sys.modules["diffusers"].AutoencoderKL = object
    spec = importlib.util.spec_from_file_location("ref_mt_vae", os.path.join(REF, "avatars/musetalk/models/vae.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    import torchvision.transforms as transforms
    v = object.__new__(ref.VAE)
    v._resized_img = 256
    v._mask_tensor = v.get_mask_tensor()
    v.transform = transforms.Normalize(mean=[0.5, 0.5, 0.5], std=[0.5, 0.5, 0.5])
    v.scaling_factor = 0.18215
    g = torch.Generator().manual_seed(23)
    sample = torch.randn(2, 3, 64, 48, generator=g) * 0.8                      # decoder output, partly outside [-1, 1]

    class FakeVae:
        device = torch.device("cpu")
        dtype = torch.float32

        def decode(self, z):
            return types.SimpleNamespace(sample=sample)
    v.vae = FakeVae()
    rng = np.random.default_rng(23)
    img = rng.integers(0, 256, (256, 256, 3), dtype=np.uint8)
    pre_full = v.preprocess_img(img, half_mask=False).numpy()
    pre_half = v.preprocess_img(img, half_mask=True).numpy()
    post = v.decode_latents(torch.zeros(2, 4, 8, 6))
    np.savez_compressed(os.path.join(HERE, "vae_glue_golden.npz"), seed=np.int64(23),
                        pre_full_crc=np.uint32(zlib.crc32(np.ascontiguousarray(pre_full).tobytes())),
                        pre_half_crc=np.uint32(zlib.crc32(np.ascontiguousarray(pre_half).tobytes())),
                        pre_full_sub=pre_full[0, :, ::37, ::41], pre_half_sub=pre_half[0, :, ::37, ::41],
                        post=np.ascontiguousarray(post))
    print("vae glue golden ok", pre_full.shape, post.shape, post.dtype)


def make_mel_windows():
    """Window starts / tail clamping of the Wav2Lip audio features from the reference's OWN MelASR.run_step
    (avatars/audio_features/mel.py:34-67), imported by path with a stub for the absent `librosa` and with
    audio.melspectrogram replaced by a fake whose value IS the mel column index (80 x (1 + N // 200), librosa's centred
    framing): the chunks the reference code queues then spell out exactly which columns each video frame gets."""
    sys.path.insert(0, os.path.join(HERE, ".."))
    import stubs
    stubs.install()
    sys.path.insert(0, REF)
    sys.modules["avatars"].__path__ = [os.path.join(REF, "avatars")]
    for k in [k for k in sys.modules if k.startswith("avatars.audio_features")]:
        del sys.modules[k]                                            # drop stubs a previous generator may have planted
    lib = types.ModuleType("librosa")
    lib.filters = types.ModuleType("librosa.filters")
    sys.modules.setdefault("librosa", lib)
    sys.modules.setdefault("librosa.filters", lib.filters)
    import importlib as il
    mel_mod = il.import_module("avatars.audio_features.mel")        # the reference file itself (+ real base_asr, real audio.py)
    audio = il.import_module("avatars.wav2lip.audio")
    audio.melspectrogram = lambda wav: np.tile(np.arange(1 + len(wav) // 200, dtype=np.float32), (80, 1))
    out = {}
    cfgs = [(16, 10, 10, 25), (4, 10, 10, 25), (1, 10, 10, 25), (8, 6, 4, 25), (4, 10, 10, 50), (2, 4, 4, 25), (32, 10, 10, 25)]
    for B, l, r, fps in cfgs:
        asr = mel_mod.MelASR(stubs.Opt(batch_size=B, l=l, r=r, fps=fps), None)
        for i in range(l + r + 2 * B):
            asr.put_audio_frame(np.full(320, float(i), np.float32), {})
        asr.warm_up()                                                 # l + r chunks of context (base_asr.py:76-82)
        asr.run_step()                                                # 2B more chunks -> B windows
        chunks = asr.feat_queue.get_nowait()
        assert len(chunks) == B and all(c.shape == (80, 16) for c in chunks), [c.shape for c in chunks]
        out[f"mel_B{B}_l{l}_r{r}_fps{fps}"] = np.asarray([c[0] for c in chunks], np.int32)      # (B, 16) column indices
    np.savez_compressed(os.path.join(HERE, "mel_window_golden.npz"), cfgs=np.asarray(cfgs, np.int32), **out)
    print("mel window golden ok", {k: v[:, 0].tolist()[:5] for k, v in out.items()})


def make_mel_chain():
    """audio.melspectrogram from the reference's OWN audio.py + hparams.py (avatars/wav2lip/audio.py:20-23, 45-51, 92-122;
    hparams.py:33-73): pre-emphasis, dB conversion, ref level, symmetric normalisation and clipping, the mel-basis arguments
    and the stft arguments are the reference's code and constants.  Only the two functions of the ABSENT librosa are
    substituted — librosa.stft and librosa.filters.mel — by the oracle's restatements, which assert the arguments the
    reference passes.  Narrows "parity unpinned" for the Wav2Lip mel to exactly those two third-party functions."""
    from oracle import mel_ref
    sys.path.insert(0, REF)
    seen = {}

    def fake_stft(y, n_fft, hop_length, win_length):
        seen["stft"] = (int(n_fft), int(hop_length), int(win_length))
        assert seen["stft"] == (800, 200, 800), seen["stft"]
        return mel_ref.stft_mag(np.asarray(y, np.float64))             # |D|; the reference takes np.abs() of it

    def fake_mel(sr, n_fft, n_mels, fmin, fmax):
        seen["mel"] = (float(sr), int(n_fft), int(n_mels), float(fmin), float(fmax))
        assert seen["mel"] == (16000.0, 800, 80, 55.0, 7600.0), seen["mel"]
        return mel_ref.mel_basis()

    lib = types.ModuleType("librosa")
    lib.stft = fake_stft
    lib.filters = types.ModuleType("librosa.filters")
    lib.filters.mel = fake_mel
    sys.modules["librosa"], sys.modules["librosa.filters"] = lib, lib.filters
    pk = types.ModuleType("refw2l")
    pk.__path__ = [os.path.join(REF, "avatars/wav2lip")]
    sys.modules["refw2l"] = pk
    import importlib as il
    audio = il.import_module("refw2l.audio")                           # the reference file (relative import of .hparams works)
    rng = np.random.default_rng(77)
    t = np.arange(16640) / 16000.0
    # loud tone (upper clip), quiet noise, an impulse, then digital silence (lower clip at -4)
    pcm = (0.95 * np.sin(2 * np.pi * 1000 * t) * (t < 0.3) + 0.01 * rng.standard_normal(t.size) * ((t >= 0.3) & (t < 0.7)) +
           0.9 * (np.abs(t - 0.8) < 0.001)).astype(np.float32)
    mel = np.asarray(audio.melspectrogram(pcm), np.float64)
    assert mel.shape == (80, 84) and "stft" in seen and "mel" in seen
    np.savez_compressed(os.path.join(HERE, "mel_chain_golden.npz"), pcm=pcm, mel=mel)
    print("mel chain golden ok", mel.shape, float(mel.min()), float(mel.max()), float((mel == -4).mean()))


def make_musereal():
    """What the reference's OWN MuseReal.inference_batch (avatars/musetalk_avatar.py:130-152) feeds the UNet and how it
    returns the result: module imported by path (heavy imports stubbed, real utils.image / PositionalEncoding), instance
    built without __init__, UNet and VAE replaced by recorders.  Pins the latent gather order (mirror_index), the dtype
    / order of the positional encoding and the timestep argument that the oracle and the engine reproduce."""
    sys.path.insert(0, os.path.join(HERE, ".."))
    import stubs
    stubs.install()
    sys.path.insert(0, REF)
    sys.modules["avatars"].__path__ = [os.path.join(REF, "avatars")]
    spec = importlib.util.spec_from_file_location("utils.image", os.path.join(REF, "utils/image.py"))
    m = importlib.util.module_from_spec(spec)
    sys.modules["utils.image"] = m
    spec.loader.exec_module(m)
    dev = types.ModuleType("utils.device")
    dev.initialize_device = lambda: "cpu"
    sys.modules["utils.device"] = dev
    av = types.ModuleType("av")
    av.AudioFrame = av.VideoFrame = object
    sys.modules["av"] = av
    for name, attrs in (("avatars.musetalk.utils", ()), ("avatars.musetalk.utils.utils", ("get_file_type", "get_video_fps", "datagen", "load_all_model")),
                        ("avatars.musetalk.whisper", ()), ("avatars.musetalk.whisper.audio2feature", ("Audio2Feature",)),
                        ("avatars.audio_features", ()), ("avatars.audio_features.whisper", ("WhisperASR",))):
        mod = types.ModuleType(name)
        mod.__path__ = []
        for a in attrs:
            setattr(mod, a, object)
        sys.modules[name] = mod
    fake = types.ModuleType("diffusers")
    fake.UNet2DConditionModel = fake.AutoencoderKL = object
    sys.modules["diffusers"] = fake
    spec = importlib.util.spec_from_file_location("ref_mt_unet2", os.path.join(REF, "avatars/musetalk/models/unet.py"))
    unet_mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(unet_mod)
    spec = importlib.util.spec_from_file_location("ref_musetalk_avatar", os.path.join(REF, "avatars/musetalk_avatar.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)

    seen = {}

    class FakeModel:
        dtype = torch.float32

        def __call__(self, latents, timesteps, encoder_hidden_states=None):
            seen["latents"], seen["timesteps"], seen["ctx"] = latents.clone(), timesteps, encoder_hidden_states.clone()
            return types.SimpleNamespace(sample=latents[:, :4] * 2.0 + 1.0)

    class FakeVae:
        def decode_latents(self, z):
            seen["decoded_from"] = z.clone()
            return z.numpy()

    B, n = 5, 3
    g = torch.Generator().manual_seed(41)
    lat_list = [torch.randn(1, 8, 4, 4, generator=g) for _ in range(n)]
    aud = [torch.randn(50, 384, generator=g).numpy() for _ in range(B)]
    mr = object.__new__(ref.MuseReal)
    mr.input_latent_list_cycle, mr.batch_size = lat_list, B
    mr.unet = types.SimpleNamespace(device="cpu", model=FakeModel())
    mr.vae, mr.pe, mr.timesteps = FakeVae(), unet_mod.PositionalEncoding(d_model=384), torch.tensor([0])
    index = 4
    out = mr.inference_batch(index, aud)
    np.savez_compressed(os.path.join(HERE, "musereal_golden.npz"), seed=np.int64(41), index=np.int64(index), batch=np.int64(B), n=np.int64(n),
                        latents=seen["latents"].numpy(), ctx_sub=seen["ctx"].numpy()[:, ::7, ::11], timesteps=seen["timesteps"].numpy(),
                        out=np.asarray(out))
    print("musereal golden ok", tuple(seen["latents"].shape), tuple(seen["ctx"].shape), seen["timesteps"])


def make_lipreal():
    """a4 + a5 + a6 as ONE piece of reference code: LipReal.inference_batch and LipReal.paste_back_frame
    (avatars/wav2lip_avatar.py:116-147) executed from the reference's own module (imported by path; `av`, MelASR,
    BaseAvatar and utils.device are stubbed, utils.image and the Wav2Lip network are the real reference files) on an
    instance built without __init__.  Pins the oracle's glue: mirror_index gather, lower-half mask, /255 in float64,
    NCHW float32, x255, astype(uint8) truncation, cv2.resize into the bbox."""
    import zlib
    sys.path.insert(0, os.path.join(HERE, ".."))
    import stubs
    stubs.install()
    sys.path.insert(0, REF)
    sys.modules["avatars"].__path__ = [os.path.join(REF, "avatars")]          # real sub-packages (avatars.wav2lip.models) resolve
    for name, rel in (("utils.image", "utils/image.py"),):
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
    dev = types.ModuleType("utils.device")
    dev.initialize_device = lambda: "cpu"
    sys.modules["utils.device"] = dev
    av = types.ModuleType("av")
    av.AudioFrame = av.VideoFrame = object
    sys.modules["av"] = av
    af = types.ModuleType("avatars.audio_features")
    af.__path__ = []
    melmod = types.ModuleType("avatars.audio_features.mel")
    melmod.MelASR = object
    sys.modules["avatars.audio_features"], sys.modules["avatars.audio_features.mel"] = af, melmod
    spec = importlib.util.spec_from_file_location("ref_wav2lip_avatar", os.path.join(REF, "avatars/wav2lip_avatar.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)

    B, n = 3, 2                                                       # batch 3 over a 2-frame avatar: mirror_index wraps and reverses
    sd = R.synth_state_dict(0)
    mel, img = R.synth_inputs(n, seed=31)
    faces = list((img[:, 3:6].permute(0, 2, 3, 1).numpy() * 255.0).round().astype(np.uint8))
    rng = np.random.default_rng(31)
    frames = [rng.integers(0, 256, (120, 160, 3), dtype=np.uint8) for _ in range(n)]
    coords = [(10, 100, 20, 150), (5, 69, 30, 94)]                    # (y1, y2, x1, x2): a stretch and a 64x64 down-scale
    melB = np.tile(mel.numpy().reshape(n, 80, 16), (2, 1, 1))[:B]
    net = ref.Wav2Lip()
    net.load_state_dict(sd, strict=True)
    net.eval()
    lip = object.__new__(ref.LipReal)
    lip.face_list_cycle, lip.frame_list_cycle, lip.coord_list_cycle = faces, frames, coords
    lip.batch_size, lip.model = B, net
    index = 1
    pred = lip.inference_batch(index, list(melB))
    pasted = [lip.paste_back_frame(pred[i], ref.mirror_index(n, index + i)) for i in range(B)]
    crops = {}
    for i in range(B):                                                # only the pasted rectangle: the rest of the frame is the seeded input
        y1, y2, x1, x2 = coords[ref.mirror_index(n, index + i)]
        crops[f"crop{i}"] = pasted[i][y1:y2, x1:x2].copy()
        outside = pasted[i].copy()
        outside[y1:y2, x1:x2] = frames[ref.mirror_index(n, index + i)][y1:y2, x1:x2]
        assert np.array_equal(outside, frames[ref.mirror_index(n, index + i)])
    # CPU conv kernels pick different blockings per batch size / thread count, so float results move in the 5th digit between
    # runs: the fixture keeps values (compared with tolerances), not checksums
    np.savez_compressed(os.path.join(HERE, "lipreal_golden.npz"), seed=np.int64(31), index=np.int64(index), batch=np.int64(B),
                        coords=np.asarray(coords, np.int32), pred_sub=pred[:, ::8, ::8, :].astype(np.float32),
                        pred_u8_sub=pred.astype(np.uint8)[:, ::4, ::4, :], **crops)
    print("lipreal golden ok", pred.shape, pred.dtype, float(pred.mean()))


def make_ultralight():
    """SURVEY 8 row f4: pins oracle/ultralight_ref.py to the reference's own code (see the module docstring)."""
    sys.path.insert(0, os.path.join(HERE, ".."))
    import stubs
    stubs.install()
    from oracle import ultralight_ref as U
    sys.path.insert(0, REF)
    sys.modules["avatars"].__path__ = [os.path.join(REF, "avatars")]
    spec = importlib.util.spec_from_file_location("utils.image", os.path.join(REF, "utils/image.py"))
    m = importlib.util.module_from_spec(spec)
    sys.modules["utils.image"] = m
    spec.loader.exec_module(m)
    dev = types.ModuleType("utils.device")
    dev.initialize_device = lambda: "cpu"
    sys.modules["utils.device"] = dev
    av = types.ModuleType("av")
    av.AudioFrame = av.VideoFrame = object
    sys.modules["av"] = av
    for name, attrs in (("avatars.audio_features", ()), ("avatars.audio_features.hubert", ("HubertASR",)),
                        ("avatars.ultralight.audio2feature", ("Audio2Feature",))):
        mod = types.ModuleType(name)
        mod.__path__ = []
        for a in attrs:
            setattr(mod, a, object)
        sys.modules[name] = mod
    spec = importlib.util.spec_from_file_location("ref_ultralight_avatar", os.path.join(REF, "avatars/ultralight_avatar.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)

    # (1) the network
    sd = U.synth_state_dict(0)
    img, audio, _faces = U.synth_inputs(2, seed=9)
    net = ref.Model(6, "hubert")
    net.load_state_dict(sd, strict=True)
    net.eval()
    with torch.no_grad():
        out = net(img, audio).numpy()
        aud = net.audio_model(audio).numpy()
    # (2) the glue: batch 3 over a 2-frame avatar (mirror_index wraps and reverses)
    B, n, index = 3, 2, 1
    _i, audio3, faces = U.synth_inputs(3, seed=21)
    faces = list(faces[:n])
    rng = np.random.default_rng(21)
    frames = [rng.integers(0, 256, (150, 200, 3), dtype=np.uint8) for _ in range(n)]
    coords = [(20, 10, 140, 130), (30, 5, 114, 89)]                   # (x1, y1, x2, y2): 120x120 stretch-down, 84x84 = exact 2x decimation
    feats = [audio3[i].numpy().reshape(16, 1024).copy() for i in range(B)]
    lr = object.__new__(ref.LightReal)
    lr.face_list_cycle, lr.frame_list_cycle, lr.coord_list_cycle = faces, frames, coords
    lr.batch_size = B

    class OnCpu(torch.nn.Module):                                      # LightReal calls .cuda() on its inputs: CPU box
        def __init__(self, inner):
            super().__init__()
            self.inner = inner

        def forward(self, a, b):
            return self.inner(a, b)

    lr.model = OnCpu(net)
    torch.Tensor.cuda = lambda self, *a, **k: self                    # noqa: E731  (build container has no GPU)
    pred = lr.inference_batch(index, feats)
    pasted = [lr.paste_back_frame(pred[i], ref.mirror_index(n, index + i)) for i in range(B)]
    crops = {}
    for i in range(B):
        x1, y1, x2, y2 = coords[ref.mirror_index(n, index + i)]
        crops[f"crop{i}"] = pasted[i][y1:y2, x1:x2].copy()
    # (3) window rows of HubertASR.run_step (hubert.py:42-45) from the reference's own BaseASR._get_sliced_feature
    spec = importlib.util.spec_from_file_location("ref_base_asr", os.path.join(REF, "avatars/audio_features/base_asr.py"))
    ba = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ba)
    asr = object.__new__(ba.BaseASR)
    rows = {}
    for (T, Bsz, l) in ((51, 16, 10), (27, 4, 10), (19, 2, 6)):
        table = np.arange(T, dtype=np.float32)[:, None] * np.ones((1, 4), np.float32)
        chunks = asr._feature2chunks(feature_array=table, batch_size=Bsz, audio_feat_win=[4, 4], start=l / 2, feature_idx_multiplier=2)
        rows[f"rows_{T}_{Bsz}_{l}"] = np.stack(chunks)[:, :, 0].astype(np.int64)
    np.savez_compressed(os.path.join(HERE, "ultralight_golden.npz"), out_sub=out[:, :, ::4, ::4].astype(np.float32),
                        out_u8=(out.transpose(0, 2, 3, 1) * 255.0).astype(np.uint8)[:, ::2, ::2], audio_emb=aud.reshape(2, -1)[:, ::16].astype(np.float32),
                        pred_sub=pred[:, ::4, ::4, :].astype(np.float32), pred_shape=np.asarray(pred.shape), coords=np.asarray(coords, np.int32),
                        index=np.int64(index), **crops, **rows)
    print("ultralight golden ok", out.shape, float(out.mean()), float(out.std()), pred.dtype)


def _audio_records(frames):
    """AudioFrameData list -> (types, data, userdata as JSON strings)."""
    import json
    return (np.asarray([f.type for f in frames], np.int32), np.stack([np.asarray(f.data, np.float32) for f in frames]),
            np.asarray([json.dumps(f.userdata, sort_keys=True) for f in frames]))


def _drain(q):
    return [q.get() for _ in range(q.qsize())]


def make_asr_host():
    """The reference's OWN BaseASR / WhisperASR / HubertASR (avatars/audio_features/*.py, imported by file path, feature
    extractors replaced by recorders) on the seeded event sequences of tests/test_plugin_host.py: frames pulled, queues,
    the PCM context handed to the extractor, the context buffer kept.  Pins the plugin's queue bookkeeping."""
    sys.path.insert(0, os.path.join(HERE, ".."))
    import stubs
    stubs.install()
    from test_plugin_host import _feed

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        return m

    out = {}
    base = load("ref_base_asr", "avatars/audio_features/base_asr.py")
    a = base.BaseASR(stubs.Opt(batch_size=3))                   # test_same_behaviour_as_reference_base_asr
    _feed(a, 23, np.random.default_rng(5))
    a.warm_up()
    out["base_get_type"], out["base_get_data"], out["base_get_ud"] = _audio_records([a.get_audio_frame() for _ in range(8)])
    out["base_outq"] = np.int64(a.output_queue.qsize())
    out["base_frames"] = np.stack(a.frames).astype(np.float32)

    af = types.ModuleType("avatars.audio_features")
    af.__path__ = []
    sys.modules["avatars.audio_features"] = af
    sys.modules["avatars.audio_features.base_asr"] = base
    for name in ("avatars.musetalk", "avatars.musetalk.whisper", "avatars.ultralight"):
        sys.modules.setdefault(name, types.ModuleType(name))
    for name in ("avatars.musetalk.whisper.audio2feature", "avatars.ultralight.audio2feature"):
        sys.modules[name] = types.ModuleType(name)
        sys.modules[name].Audio2Feature = object

    B = 3                                                       # test_whisper_asr_run_step_bookkeeping_matches_reference
    whisper = load("ref_whisper_asr", "avatars/audio_features/whisper.py")

    class WhisperRecorder:
        def __init__(self):
            self.calls = []

        def audio2feat(self, pcm):
            self.calls.append(np.asarray(pcm).copy())
            return np.zeros((1500, 5, 384), np.float32)

    rec = WhisperRecorder()
    w = whisper.WhisperASR(stubs.Opt(batch_size=B), None, rec)
    _feed(w, 20 + 2 * B + 2, np.random.default_rng(2))
    w.warm_up()
    w.run_step()
    assert w.feat_queue.qsize() == 1 and len(rec.calls) == 1
    out["whisper_feat_shape"] = np.asarray([np.asarray(f).shape for f in w.feat_queue.get()], np.int32)
    out["whisper_pcm"] = rec.calls[0].astype(np.float32)
    out["whisper_frames"] = np.stack(w.frames).astype(np.float32)
    out["whisper_out_type"], out["whisper_out_data"], _ = _audio_records(_drain(w.output_queue))

    hubert = load("ref_hubert_asr", "avatars/audio_features/hubert.py")   # test_hubert_asr_run_step_bookkeeping_matches_reference

    class HubertRecorder:
        def __init__(self):
            self.calls = []

        def get_hubert_from_16k_speech(self, pcm):
            self.calls.append(np.asarray(pcm).copy())
            return np.ones(((len(pcm) - 80) // 320, 1024), np.float32)

    rec = HubertRecorder()
    h = hubert.HubertASR(stubs.Opt(batch_size=B), None, rec, audio_feat_length=[4, 4])
    _feed(h, 20 + 2 * B, np.random.default_rng(4))
    h.warm_up()
    shapes = []
    for _step in range(3):
        h.run_step()
        shapes.append([np.asarray(f).shape for f in h.feat_queue.get()])
    out["hubert_feat_shapes"] = np.asarray(shapes, np.int32)
    out["hubert_pcm"] = np.stack(rec.calls).astype(np.float32)
    out["hubert_last_is_silence"] = np.bool_(h.last_is_silence)
    out["hubert_frames"] = np.stack(h.frames).astype(np.float32)
    out["hubert_out_type"], out["hubert_out_data"], _ = _audio_records(_drain(h.output_queue))
    np.savez_compressed(os.path.join(HERE, "asr_host_golden.npz"), **out)
    print("asr host golden ok", {k: v.shape for k, v in out.items()})


def make_mt_blend():
    """The reference's OWN get_image_blending (avatars/musetalk/myutil.py) driven as MuseReal.paste_back_frame does, on the
    seeded frame / prediction / masks of tests/test_oracle_paste.py::test_musetalk_blend_matches_cv2_and_reference_function."""
    import cv2
    sys.path.insert(0, os.path.join(HERE, ".."))
    from test_oracle_paste import mt_blend_case
    spec = importlib.util.spec_from_file_location("ref_myutil", os.path.join(REF, "avatars/musetalk/myutil.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    frame, pred, bbox, crop, masks = mt_blend_case()
    x1, y1, x2, y2 = bbox
    want = [ref.get_image_blending(frame.copy(), cv2.resize(pred, (x2 - x1, y2 - y1)), bbox, m, crop) for m in masks]
    np.savez_compressed(os.path.join(HERE, "mt_blend_golden.npz"), want=np.stack(want))
    print("mt blend golden ok", np.stack(want).shape)


if __name__ == "__main__":
    if not os.path.isfile(os.path.join(REF, "avatars", "base_avatar.py")):
        sys.exit("set LTB_REFERENCE to a LiveTalking checkout")
    make_w2l()
    make_paste()
    make_mel()
    make_slices()
    make_pe()
    make_vae_glue()
    make_lipreal()
    make_mel_windows()
    make_mel_chain()
    make_musereal()
    make_ultralight()
    make_asr_host()
    make_mt_blend()
