"""What the n-tuple GPU tests share: the ``ops`` fixture (the library built and loaded) and the CUDA device."""

from __future__ import annotations

import pytest
import torch


@pytest.fixture(scope="module")
def ops():
    from ml2048_b200 import _lib, build, ops

    build.build()
    _lib.load()
    return ops


def _gpu():
    assert torch.cuda.is_available()
    return torch.device("cuda")
