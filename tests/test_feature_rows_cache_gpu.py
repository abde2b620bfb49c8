"""functional.feature_rows caches the last map's channels-last rows; a new map must never get a freed map's rows, even when
the allocator places it at the freed map's address with the same shape and version."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_new_map_at_a_reused_address_gets_its_own_rows(lib):
    from meshrcnn_b200 import functional as F_
    g = torch.Generator().manual_seed(0)
    a_h, b_h = torch.randn(2, 8, 6, 6, generator=g), torch.randn(2, 8, 6, 6, generator=g)
    want = lambda m: m.permute(0, 2, 3, 1).reshape(-1, 8)
    a = a_h.cuda()
    assert torch.equal(F_.feature_rows(a).cpu(), want(a_h))
    assert F_.feature_rows(a) is F_.feature_rows(a)                       # the same map: one conversion
    ptr = a.data_ptr()
    del a
    b = b_h.cuda()
    assert b.data_ptr() == ptr and b._version == 0                          # the case the cache must not confuse
    assert torch.equal(F_.feature_rows(b).cpu(), want(b_h))
