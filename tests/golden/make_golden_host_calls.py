"""Generates tests/golden/golden_host_calls.npz: the call patterns of tests/test_host_vs_reference.py and of
test_live_against_the_unmodified_reference_modules in tests/test_post_decode_host.py, which compare the product with the
reference wrapper and the reference's utils/audio_utils.py.

Where the reference is installed (oracle/reference_wrapper.py, oracle/post_decode_oracle.py) the vectors are its outputs.
Without it they are recorded from the product tokenizer and the oracle restatement of the utilities, both of which the
tests above and tests/test_oracle_golden.py / tests/test_post_decode_host.py hold to the reference's own golden vectors.
The npz key ``source`` says which.                                  python tests/golden/make_golden_host_calls.py
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import rca_b200_loader  # noqa: E402,F401
import realtime_codec_agent_b200 as pkg  # noqa: E402
from oracle import post_decode_oracle as po  # noqa: E402
from oracle.magicodec_oracle import OracleGenerator  # noqa: E402
from oracle.reference_wrapper import load_reference_audio_tokenizer, reference_available  # noqa: E402
from tests import test_host_vs_reference as hv, test_post_decode_host as pd  # noqa: E402
from tests.golden.make_golden import save_npz_lzma  # noqa: E402
from tests.golden_calls import to_golden  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def main():
    torch.manual_seed(0)
    ref = reference_available() and po.reference_available()
    Tok = load_reference_audio_tokenizer() if ref else pkg.AudioTokenizer
    model = OracleGenerator(pkg.TINY_SPEC, pkg.init_random_weights(pkg.TINY_SPEC, seed=0))
    out = {"source": np.array("reference" if ref else "product tokenizer + oracle restatement of the utilities")}
    for channels in hv.CHANNELS:
        for chunk_ms in hv.CHUNK_MS:
            out.update(to_golden(hv.streaming_calls(Tok, model, channels, chunk_ms), f"stream_c{channels}_{chunk_ms}ms"))
    out.update(to_golden(hv.int16_calls(Tok, model), "int16"))

    utils = {k: getattr(po.load_reference_module("utils.audio_utils"), k) for k in po.RESTATED_UTILS} if ref else po.RESTATED_UTILS
    out.update(to_golden(pd.util_calls(utils), "post_utils", sample=False))
    model, our_tok, s = pd.oracle_model_tokenizer_and_codes()
    chain = po.OracleOutputChain(Tok(codec_model=model, device="cpu") if ref else our_tok, 0.1, 0.02, 0.05, utils=utils)
    out.update(to_golden(pd.chain_calls(chain.step, lambda: chain.history, s), "post_chain"))
    path = os.path.join(OUT, "golden_host_calls.npz")
    save_npz_lzma(path, out)
    print(path, os.path.getsize(path), "bytes,", len(out), "arrays, source:", out["source"])


if __name__ == "__main__":
    main()
