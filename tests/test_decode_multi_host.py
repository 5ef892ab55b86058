"""Host-side checks of the multi-token decode entry (pli_decode_fwd_multi): argument rejection before any launch and the
split-count rule; no GPU needed."""
import ctypes

import pytest
import torch

import physics_llm_inference_b200 as pli
from physics_llm_inference_b200 import _lib


def _call(q_len, q_strides, o_strides, Hq=8, Hkv=2, D=128):
    lib = _lib.load()
    dummy = ctypes.c_void_p(256)               # never dereferenced: the arguments are rejected first
    return lib.pli_decode_fwd_multi(dummy, dummy, dummy, None, dummy, dummy, None, 2, Hq, Hkv, q_len, D, 100, 0, 0, 0,
                                    2, _lib.i64(*q_strides), _lib.i64(1024, 0, 256, 128), _lib.i64(*o_strides), 0.1,
                                    _lib.PLI_BF16, 1, dummy, 1 << 20, None)


def test_multi_entry_rejects_before_launch():
    n0 = _lib.launch_count()
    assert _call(17, (8 * 17 * 128, 17 * 128, 128), (8 * 17 * 128, 17 * 128, 128)) == -2      # PLI_ERR_UNSUPPORTED
    assert b"16" in _lib.load().pli_last_error()
    assert _call(0, (1024, 128, 128), (1024, 128, 128)) == -1                                # PLI_ERR_INVALID
    # o's head stride must be q_len * its token stride (q is read through any strides)
    assert _call(4, (8 * 4 * 128, 4 * 128, 128), (8 * 4 * 128, 128, 8 * 128)) == -1
    assert b"o needs" in _lib.load().pli_last_error()
    assert _lib.launch_count() == n0


def test_split_count_counts_row_chunks():
    # C3 with 8 tokens: 32 rows per KV head = two 16-row chunks per unit
    assert pli.decode_num_splits(1, 8, 32768, group=4, q_len=8) == pli.decode_num_splits(1, 16, 32768)
    assert pli.decode_num_splits(1, 8, 32768, group=4, q_len=4) == pli.decode_num_splits(1, 8, 32768)
    assert pli.decode_num_splits(1, 8, 32768, group=32) == pli.decode_num_splits(1, 8, 32768)
    lib = _lib.load()
    # one token: exactly pli_decode_fwd's choice, also for G > 16
    assert lib.pli_decode_num_splits_multi(1, 8 * 32, 8, 1, 32768) == lib.pli_decode_num_splits(1, 8, 32768)
    assert lib.pli_decode_num_splits_multi(1, 32, 8, 8, 32768) == lib.pli_decode_num_splits(1, 16, 32768)


def test_multi_token_python_rejections_without_gpu():
    q = torch.zeros(1, 2, 4, 16)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pli.flash_decode(q, torch.zeros(1, 8, 2, 16), torch.zeros(1, 8, 2, 16), 8)
    with pytest.raises(ValueError, match="tokens_per_step"):
        pli.DecodeGraphRunner(torch.zeros(1, 8, 2, 16), torch.zeros(1, 8, 2, 16), 2, tokens_per_step=17)
