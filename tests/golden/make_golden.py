"""Generates tests/golden/*.npz by running the UNMODIFIED reference wrapper
(/root/reference/realtime_codec_agent/audio_tokenizer.py, loaded by oracle/reference_wrapper.py)
around OracleGenerator with the seeded weights of realtime_codec_agent_b200.weights.

Run in the build container only (needs /root/reference):   python tests/golden/make_golden.py
The fixtures pin (a) the oracle restatement + host-side string/length arithmetic against the
reference wrapper's own behaviour and (b) the inputs/outputs the GPU parity tests replay.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import rca_b200_loader  # noqa: E402,F401
import realtime_codec_agent_b200 as pkg  # noqa: E402
from oracle.magicodec_oracle import OracleGenerator  # noqa: E402
from oracle.reference_wrapper import load_reference_audio_tokenizer  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def save_npz_lzma(path: str, arrays: dict) -> None:
    """np.savez with LZMA entries: np.load reads it unchanged, and golden_tiny.npz stays under 1 MB (deflate: 1.03 MB)."""
    import io
    import zipfile
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for k, v in arrays.items():
            buf = io.BytesIO()
            np.save(buf, np.asanyarray(v))
            z.writestr(k + ".npy", buf.getvalue())


def make(spec_name: str, spec, secs: float):
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count() or 1)
    weights = pkg.init_random_weights(spec, seed=0)
    model = OracleGenerator(spec, weights)
    RefTok = load_reference_audio_tokenizer()
    n = int(secs * spec.sample_rate)
    wav0 = pkg.synth_audio(n, seed=1234, file_id=0, channel=0).numpy()
    wav1 = pkg.synth_audio(n, seed=1234, file_id=0, channel=1).numpy()
    out = {"wav0": wav0.astype(np.float16).astype(np.float32)}     # fp16-exact inputs keep the file small
    wav0 = out["wav0"]
    out["wav1"] = wav1.astype(np.float16).astype(np.float32)
    wav1 = out["wav1"]

    # mono, one-shot
    tok = RefTok(codec_model=model, device="cpu")
    out["framerate"] = np.float64(tok.framerate)
    s = tok.tokenize_audio(wav0)
    out["mono_oneshot_codes"] = np.array([ord(c) - tok.unicode_offset for c in s], dtype=np.int32)
    (sr, rec), hang, pre = tok.detokenize_audio(s)
    out["mono_oneshot_wav"] = rec.astype(np.float32)
    # mono, chunked 0.1 s (the normative offline encode, audio_tokenizer.py:52-65)
    tok.reset_context()
    s = tok.chunked_tokenize_audio(wav0, 0.1)
    out["mono_chunked_codes"] = np.array([ord(c) - tok.unicode_offset for c in s], dtype=np.int32)
    # streaming decode of those codes in 0.1 s (5 char) chunks with a 320-sample preroll
    tok.reset_context()
    pieces, pre = [], 320
    for i in range(0, len(s), 5):
        (sr, rec), hang, pre_left = tok.detokenize_audio(s[i:i + 5], preroll_samples=320)
        pieces.append(rec[-1600:])
    out["mono_stream_decode_wav"] = np.concatenate(pieces).astype(np.float32)
    # the 0.58 s truncation quirk and a 20 ms chunk
    tok.reset_context()
    out["len_058"] = np.int64(len(tok.tokenize_audio(wav0[: int(0.58 * 16000)])))
    out["len_002"] = np.int64(len(tok.tokenize_audio(wav0[:320])))
    # stereo chunked 0.1 s
    tok2 = RefTok(codec_model=model, num_channels=2, device="cpu")
    st = np.stack([wav0, wav1])
    s2 = tok2.chunked_tokenize_audio(st, 0.1)
    out["stereo_chunked_codes"] = np.array([ord(c) - tok2.unicode_offset for c in s2], dtype=np.int32)
    (sr, rec2), hang, pre = tok2.detokenize_audio(s2[:201])     # odd length -> hanging code dropped
    out["stereo_decode_wav"] = rec2.astype(np.float32)
    out["stereo_hanging"] = np.array([ord(c) for c in hang], dtype=np.int32)

    # raw network taps for the GPU parity tests (window of the last 2.0 s, batch of 2)
    x = torch.from_numpy(np.stack([wav0[-32000:], wav1[-32000:]]))
    with torch.no_grad():
        z_e = model.encoder(model.pad_audio(x))
        z_q, idx, margin = model.quantizer.inference(z_e, return_margin=True)
        rec = model.decoder(z_q)
    out["tap_z_e"] = z_e.numpy()
    out["tap_idx"] = idx.numpy().astype(np.int32)
    out["tap_margin"] = margin.numpy()
    out["tap_rec"] = rec.numpy()[:, 0]
    save_npz_lzma(os.path.join(OUT, f"golden_{spec_name}.npz"), out)
    print(spec_name, {k: (v.shape if hasattr(v, "shape") else v) for k, v in out.items()})


if __name__ == "__main__":
    make("tiny", pkg.TINY_SPEC, 3.0)
    make("mid", pkg.MID_SPEC, 2.5)
