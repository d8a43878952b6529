"""pb_mlp_update_fused through the C ABI, stage by stage (tests/experimental/check_mlp_update_fused.py has the details):
forward UMMA vs TF32-truncated fp64 math, dOut / statistics vs pb_ppo_loss on the kernel's own head outputs, dPre, and every
gradient section vs fp64 products of the kernel's own dumps; then the same launch without dumps.
Shapes: one tile, a ragged tile count, more tiles than SMs, several slabs with gaps (the zero-copy minibatch layout), 1 / 4 / 7
actions.  Reference of the math: /root/reference/clean_pufferl.py:186-244 with the policy of pufferlib/models.py:12-62."""
import os
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'experimental'))

pytestmark = pytest.mark.gpu

SHAPES = [(128, 1, 128, 4, 1), (1000, 1, 1000, 4, 2), (148 * 128 * 2 + 77, 1, 148 * 128 * 2 + 77, 7, 3), (300, 2, 1000, 1, 4),
          (4096, 4, 16384, 4, 5)]


@pytest.mark.parametrize('slab_rows,n_slabs,slab_stride,n_act,seed', SHAPES)
def test_fused_update_kernel_stages(slab_rows, n_slabs, slab_stride, n_act, seed):
    import check_mlp_update_fused as cf
    assert cf.case(slab_rows, n_slabs, slab_stride, n_act, seed)
