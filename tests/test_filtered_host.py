"""Host side of filtered evaluation (CPU only): the driver flag, and the refusals that need no device."""
import ctypes

import numpy as np
import pytest
import torch

import gcn_vae_b200 as K


def test_filtered_flag_parses_and_defaults_to_off():
    p = K.link_predict.build_parser()
    assert p.parse_args(["-d", "toy"]).filtered is False
    assert p.parse_args(["-d", "toy", "--filtered"]).filtered is True


def test_filter_index_refuses_cpu():
    known = np.array([[0, 0, 1], [1, 0, 2]])
    with pytest.raises(RuntimeError, match="CUDA"):
        K.utils.FilterIndex(known, 3, 1, "cpu")
    with pytest.raises(RuntimeError, match="CUDA"):
        K.utils.FilterIndex(torch.from_numpy(known), 3, 1, torch.device("cpu"))


def test_filter_table_refuses_keys_wider_than_64_bits():
    """2 bits(N) + bits(R) > 64 is refused before any device work: N = 2^31 - 1 needs 31 bits, R = 8 needs 3."""
    lib = K._lib.lib()
    rc = lib.kg_filter_table(None, 0, 2 ** 31 - 1, 8, 0, None, None, None, 0, None)
    assert rc == -1 and b"64" in lib.kg_last_error()
    assert lib.kg_filter_table(None, 0, 10, 4, 2, None, None, None, 0, None) == -1     # no such direction
