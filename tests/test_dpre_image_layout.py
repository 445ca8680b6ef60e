"""The 16-bit dPre image layout of the tensor-core backward (csrc/attn.cu, attn_bwd_img_kernel): the image builder the
consumer tests use (test_gpu_tc.dpre_image) and the decoder the producer tests use
(test_gpu_tc_backward.decode_dpre_image) are exact inverses.  CPU only."""
import numpy as np
import pytest

from test_gpu_tc import dpre_image, round16
from test_gpu_tc_backward import decode_dpre_image


@pytest.mark.parametrize('L', [1, 31, 32, 63])
@pytest.mark.parametrize('F', [16, 48, 272, 400, 496, 512])
@pytest.mark.parametrize('fp16', [1, 0])
def test_decode_inverts_dpre_image(L, F, fp16):
    N = 3
    g = np.random.default_rng(L * 1000 + F + fp16)
    x = round16(g.standard_normal((N, L, F)).astype(np.float32), fp16)
    img = dpre_image(x, fp16)
    slot, ngh = (32 if L <= 31 else 64), (F // 2 + 63) // 64
    assert img.size * 2 == N * 2 * ngh * slot * 128          # lstur_tc_dpre_img_bytes(N, L, F)
    assert np.array_equal(decode_dpre_image(img, N, L, F, fp16), x.astype(np.float64))
