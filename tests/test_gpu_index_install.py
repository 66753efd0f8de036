"""Installing an index: build_index, build_index_trim and upload_sa share one install, so a forced 32-bit width is refused
alike by all of them for a strand of n+1 >= 2^32-2."""
import numpy as np
import pytest

import asgart_b200 as ab
from asgart_b200 import _lib

pytestmark = pytest.mark.gpu


def test_upload_sa_refuses_32_bit_width_for_long_strand():
    n1 = 2**32 - 1   # 'A' * (2**32 - 2) + '$': 4 GiB of host memory, 6 GiB on the device (text and packed image)
    strand = np.full(n1, ord("A"), dtype=np.uint8)
    strand[-1] = ord("$")
    with ab.Context(0) as ctx:
        ctx.set_index_bits(32)
        ctx.load_strand(strand)
        del strand
        with pytest.raises(ab.AsgartB200Error) as built:
            ctx.build_index()
        assert built.value.code == _lib.EINVAL
        # zero pages, mapped lazily: a refused upload reads none of the 32 GiB, one that narrowed the entries reads them all
        sa = np.zeros(n1, np.int64)
        rc = ctx.L.asgart_b200_ctx_upload_sa(ctx.h, sa.ctypes.data)
        assert rc == _lib.EINVAL
        assert ctx.L.asgart_b200_ctx_last_error(ctx.h).decode() == "32-bit indices need n+1 < 2^32-2"
        assert str(built.value).endswith("32-bit indices need n+1 < 2^32-2")
