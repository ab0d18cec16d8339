"""Chunk-and-average long-audio mode (SURVEY.md §8f rank 4): wespeaker_b200.speaker_engine against the literal restatement
of runtime/core/speaker/speaker_engine.cc in oracle/speaker_engine_py.py."""
import numpy as np
import pytest
import torch

from oracle import fbank_np, models_torch, speaker_engine_py as ref
from wespeaker_b200 import synthetic as syn
from wespeaker_b200.speaker_engine import SpeakerEngine, chunk_frame_index


@pytest.mark.parametrize("T,n", [(1, 198), (7, 198), (66, 198), (99, 198), (100, 198), (197, 198), (198, 198), (199, 198),
                                 (396, 198), (500, 198), (1000, 198), (5, 3), (3, 5), (0, 198)])
def test_chunk_index_matches_cpp_vector_logic(T, n):
    per_chunk_samples = 400 + (n - 1) * 160
    assert ref.num_chunk_frames(per_chunk_samples) == n
    want = ref.extract_feature(list(range(T)), per_chunk_samples)
    got = chunk_frame_index(T, n)
    assert got.shape == (len(want), n)
    assert [list(r) for r in got] == want


@pytest.mark.parametrize("nsamp", [9000, 32000, 50000, 100000])
def test_engine_host_logic_with_oracle_frontend_and_model(nsamp):
    """Whole SpeakerEngine with the CPU oracles injected for fbank and the model: isolates the chunk / CMN / average logic."""
    name = "ECAPA_TDNN_c512"
    sd = syn.make_state_dict(name, seed=0)
    fwd = lambda feats: models_torch.forward(name, sd, torch.as_tensor(feats, dtype=torch.float32))
    wav = syn.make_wavs(1, nsamp, seed=7)[0]
    fb = lambda w: torch.from_numpy(fbank_np.fbank(np.asarray(w[0], dtype=np.float32), window_type="hamming"))
    eng = SpeakerEngine(model=None, embedding_size=192, samples_per_chunk=32000, fbank_fn=fb, embed_fn=fwd)
    got = eng.extract_embedding(wav)
    frames = list(fbank_np.fbank(wav.astype(np.float32), window_type="hamming"))
    want = ref.extract_embedding(frames, 32000, lambda c: fwd(c[None])[0].numpy())
    assert got.shape == (192,)
    assert np.linalg.norm(got - want) / np.linalg.norm(want) < 1e-5
    assert SpeakerEngine.cosine_similarity(got, want) == pytest.approx(1.0, abs=1e-6)
    assert SpeakerEngine.cosine_similarity(got, -want) == pytest.approx(0.0, abs=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("nsamp", [9000, 50000, 163840])
def test_engine_gpu_matches_oracle(nsamp):
    from wespeaker_b200.models import from_synthetic
    name = "ECAPA_TDNN_c512"
    m = from_synthetic(name, 0, precision="fp32")
    wav = syn.make_wavs(1, nsamp, seed=7)[0]
    got = SpeakerEngine(m, samples_per_chunk=32000).extract_embedding(torch.from_numpy(wav))
    sd = syn.make_state_dict(name, seed=0)
    fwd = lambda feats: models_torch.forward(name, sd, torch.as_tensor(feats, dtype=torch.float32))
    frames = list(fbank_np.fbank(wav.astype(np.float32), window_type="hamming"))
    want = ref.extract_embedding(frames, 32000, lambda c: fwd(c[None])[0].numpy())
    assert np.linalg.norm(got - want) / np.linalg.norm(want) < 1e-4
    # full mode == plain extraction of the whole recording
    full = SpeakerEngine(m, samples_per_chunk=-1).extract_embedding(torch.from_numpy(wav))
    ref_full = ref.extract_embedding(frames, -1, lambda c: fwd(c[None])[0].numpy())
    assert np.linalg.norm(full - ref_full) / np.linalg.norm(ref_full) < 1e-4


# ------------------------------------------------------------------------------------------------- pinned on the reference's C++
G_REF = np.load(__import__("os").path.join(__import__("os").path.dirname(__file__), "golden", "ref_engine.npz"))


@pytest.mark.parametrize("nsamp", [9000, 20000, 32000, 50000, 80333, 163840])
def test_chunk_logic_pinned_on_compiled_reference(nsamp):
    """tests/golden/ref_engine.npz comes from the reference's own speaker_engine.cc / feature_pipeline.cc / fbank.h compiled
    into oracle/_ref (make -C oracle): which native-fbank frame every row of every chunk is.  The Python restatement
    (oracle) and the product's index builder must reproduce it exactly."""
    want = G_REF[f"chunk_index_{nsamp}"]
    T = int(G_REF[f"nframes_{nsamp}"])
    assert T == 1 + (nsamp - 400) // 160
    assert ref.extract_feature(list(range(T)), 32000) == [list(r) for r in want]
    assert np.array_equal(chunk_frame_index(T, 198), want)


@pytest.mark.parametrize("nsamp", [9000, 50000])
def test_fbank_and_apply_mean_oracles_pinned_on_compiled_reference(nsamp):
    """The numpy fbank oracle (restating torchaudio's kaldi.fbank) against the reference's NATIVE fbank twin
    (runtime/core/frontend/fbank.h: own radix-2 FFT, double-precision window) on the same int16 PCM, and ApplyMean."""
    pcm = syn.make_wavs(1, nsamp, seed=7)[0].astype(np.int16).astype(np.float32)
    mine = fbank_np.fbank(pcm, window_type="hamming")
    full = G_REF[f"full_{nsamp}"]
    assert mine.shape == full.shape
    d = np.abs(mine - full)
    print(f"fbank_np vs native fbank.h, {nsamp} samples: max {d.max():.2e} mean {d.mean():.2e}")
    assert d.max() < 5e-3 and d.mean() < 5e-5                      # log-mel units; FFT algorithm / window precision differ
    idx = G_REF[f"chunk_index_{nsamp}"]
    last = ref.apply_mean(full[idx[-1]])
    assert np.abs(last - G_REF[f"lastchunk_cmn_{nsamp}"]).max() < 2e-5


def test_cosine_similarity_pinned_on_compiled_reference():
    for a, b, want in zip(G_REF["cos_a"], G_REF["cos_b"], G_REF["cos"]):
        assert SpeakerEngine.cosine_similarity(a, b) == pytest.approx(float(want), abs=2e-6)


def test_live_compiled_reference_if_present():
    """On boxes where oracle/_ref/libref_engine.so travelled (it is built here from /root/reference and is not gpurun-ignored)
    the fixture is re-derived live: guards against a stale fixture."""
    import ctypes as C
    import os
    so = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libref_engine.so")
    if not os.path.exists(so):
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    L = C.CDLL(so)
    L.ref_extract_feature.restype = C.c_int
    L.ref_extract_feature.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.c_int)]
    L.ref_free.argtypes = [C.POINTER(C.c_float)]
    pcm = np.ascontiguousarray(syn.make_wavs(1, 9000, seed=7)[0].astype(np.int16))
    out, shape = C.POINTER(C.c_float)(), (C.c_int * 3)()
    assert L.ref_extract_feature(pcm.ctypes.data, len(pcm), 0, 0, C.byref(out), shape) == 1
    full = np.ctypeslib.as_array(out, shape=(shape[1] * shape[2],)).copy().reshape(shape[1], shape[2])
    L.ref_free(out)
    assert np.array_equal(full, G_REF["full_9000"])


@pytest.mark.gpu
@pytest.mark.parametrize("nsamp,chunk", [(50000, 32000), (9000, 32000), (50000, 0)])
def test_cpp_seam_reference_engine_with_b200_model(nsamp, chunk, tmp_path):
    """Seam B4: the reference's own C++ SpeakerEngine (compiled unmodified into oracle/_ref/libb200_seam.so) with
    wespeaker::B200SpeakerModel (csrc/runtime/b200_speaker_model.cc) in its model slot: reference fbank -> chunking ->
    ApplyMean -> virtual ExtractEmbedding -> B200 engine -> reference averaging, against the oracle model fed with the
    reference's own frames (fixture)."""
    import ctypes as C
    import os
    from wespeaker_b200.models import from_synthetic
    so = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libb200_seam.so")
    if not os.path.exists(so):
        pytest.skip("oracle/_ref/libb200_seam.so not built (make -C oracle all needs /root/reference)")
    name = "ECAPA_TDNN_c512"
    m = from_synthetic(name, 0, precision="fp32")
    flat = str(tmp_path / "model.wsb")
    m.export_flat(flat)
    L = C.CDLL(so)
    L.ref_engine_extract_with_b200.restype = C.c_int
    L.ref_engine_extract_with_b200.argtypes = [C.c_char_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
    pcm = np.ascontiguousarray(syn.make_wavs(1, nsamp, seed=7)[0].astype(np.int16))
    emb = np.zeros(192, dtype=np.float32)
    assert L.ref_engine_extract_with_b200(flat.encode(), 0, pcm.ctypes.data, len(pcm), chunk, emb.ctypes.data, 192) == 0
    sd = syn.make_state_dict(name, seed=0)
    fwd = lambda feats: models_torch.forward(name, sd, torch.as_tensor(feats, dtype=torch.float32))
    frames = list(G_REF[f"full_{nsamp}"])                      # the reference's native fbank frames of this PCM
    want = ref.extract_embedding(frames, chunk, lambda c: fwd(c[None])[0].numpy())
    rel = np.linalg.norm(emb - want) / np.linalg.norm(want)
    print(f"C++ seam nsamp {nsamp} chunk {chunk}: rel {rel:.2e}")
    assert rel < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("nsamp,chunk", [(50000, 32000), (9000, 32000), (50000, 0)])
def test_cpp_b200_speaker_model_per_chunk_matches_oracle(nsamp, chunk, tmp_path):
    """wespeaker::B200SpeakerModel (csrc/runtime/b200_speaker_model.cc, in build/libb200_model_harness.so) called through
    the virtual SpeakerModel::ExtractEmbedding, one chunk per call, with no file from outside this repository: the
    reference's native fbank frames of this PCM (fixture) are chunked and mean-normalised by the Python restatement (pinned
    above on the reference's own outputs) on both sides, and the average of the B200 embeddings is compared with the CPU
    oracle model's.  The interface is a stand-in (oracle/seam_shim), so compatibility with the real speaker_model.h is not
    checked here; test_cpp_seam_reference_engine_with_b200_model does that where the WeSpeaker sources were built."""
    import ctypes as C
    import os
    from wespeaker_b200.models import from_synthetic
    so = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "build", "libb200_model_harness.so")
    name = "ECAPA_TDNN_c512"
    m = from_synthetic(name, 0, precision="fp32")
    flat = str(tmp_path / "model.wsb")
    m.export_flat(flat)
    L = C.CDLL(so)
    L.b200_model_extract_chunks.restype = C.c_int
    L.b200_model_extract_chunks.argtypes = [C.c_char_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
    frames = list(G_REF[f"full_{nsamp}"])                      # the reference's native fbank frames of this PCM
    chunks = np.ascontiguousarray(np.stack([ref.apply_mean(c) for c in ref.extract_feature(frames, chunk)]))
    embs = np.zeros((chunks.shape[0], 192), dtype=np.float32)
    assert L.b200_model_extract_chunks(flat.encode(), 0, chunks.ctypes.data, chunks.shape[0], chunks.shape[1],
                                       chunks.shape[2], embs.ctypes.data, 192) == 0
    emb = embs.sum(axis=0) / chunks.shape[0]
    sd = syn.make_state_dict(name, seed=0)
    fwd = lambda feats: models_torch.forward(name, sd, torch.as_tensor(feats, dtype=torch.float32))
    want = ref.extract_embedding(frames, chunk, lambda c: fwd(c[None])[0].numpy())
    rel = np.linalg.norm(emb - want) / np.linalg.norm(want)
    print(f"B200SpeakerModel per chunk, nsamp {nsamp} chunk {chunk}: rel {rel:.2e}")
    assert rel < 1e-4
