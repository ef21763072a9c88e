"""CPU checks of the data-parallel fit's plumbing: the exchange-buffer layout and stage numbers the Python side uses are the
ones include/ofb_train.h declares, every stage maps to the slice it names, and sharding.DistReducer reduces and broadcasts."""
import os
import re
from types import SimpleNamespace

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_constants():
    txt = open(os.path.join(ROOT, "include", "ofb_train.h")).read()
    out = {k: int(v) for k, v in re.findall(r"#define (OFB_TRAIN_\w+) (\d+)", txt)}
    out.update({k: int(v) for k, v in re.findall(r"(OFB_STAGE_\w+) = (\d+)", txt)})
    return out


def test_python_layout_is_the_headers():
    from ofighters_b200 import _lib
    h = _header_constants()
    assert (h["OFB_TRAIN_N_BN"], h["OFB_TRAIN_STATS_FWD"], h["OFB_TRAIN_STATS_LOSS"], h["OFB_TRAIN_STATS_BWD"],
            h["OFB_TRAIN_STATS_LEN"]) == (_lib.TRAIN_N_BN, _lib.TRAIN_STATS_FWD, _lib.TRAIN_STATS_LOSS, _lib.TRAIN_STATS_BWD,
                                          _lib.TRAIN_STATS_LEN)
    assert (h["OFB_STAGE_FWD_BN"], h["OFB_STAGE_LOSS"], h["OFB_STAGE_BWD_BN"], h["OFB_STAGE_GRADS"]) == \
        (_lib.STAGE_FWD_BN, _lib.STAGE_LOSS, _lib.STAGE_BWD_BN, _lib.STAGE_GRADS)
    # forward sums, the loss pair and backward sums tile the buffer without overlap
    assert _lib.TRAIN_STATS_LOSS == _lib.TRAIN_STATS_FWD + 16 * _lib.TRAIN_N_BN
    assert _lib.TRAIN_STATS_BWD == _lib.TRAIN_STATS_LOSS + 2
    assert _lib.TRAIN_STATS_LEN == _lib.TRAIN_STATS_BWD + 16 * _lib.TRAIN_N_BN


def test_every_stage_names_its_own_slice():
    from ofighters_b200 import _lib
    from ofighters_b200.trainer import TrainerB200, len_flat
    fake = SimpleNamespace(_xstats=torch.zeros(_lib.TRAIN_STATS_LEN, dtype=torch.float64),
                           _xgrads=torch.zeros(len_flat(), dtype=torch.float32))
    seen = torch.zeros(_lib.TRAIN_STATS_LEN, dtype=torch.int32)
    for stage in range(16):
        t = TrainerB200._exchange_slice(fake, stage)
        if stage == _lib.STAGE_GRADS:
            assert t.data_ptr() == fake._xgrads.data_ptr() and t.numel() == 571730
            continue
        off = (t.data_ptr() - fake._xstats.data_ptr()) // 8
        seen[off:off + t.numel()] += 1
    assert bool((seen == 1).all())                      # 16 stages cover the 226 doubles exactly once
    with pytest.raises(Exception, match="unknown reduce stage"):
        TrainerB200._exchange_slice(fake, 16)


def test_dist_reducer_over_gloo(tmp_path):
    import torch.distributed as dist
    from ofighters_b200.sharding import DistReducer
    with pytest.raises(Exception, match="process group"):
        DistReducer()
    dist.init_process_group("gloo", init_method="file://" + str(tmp_path / "pg"), rank=0, world_size=1)
    try:
        r = DistReducer()
        assert (r.rank, r.world) == (0, 1)
        t = torch.tensor([3.0, -1.0], dtype=torch.float64)
        r.all_reduce(t)
        r.all_reduce(t, op="min")
        r.broadcast(t, src=0)
        assert t.tolist() == [3.0, -1.0]
        with pytest.raises(Exception, match="Invalid op"):
            r.all_reduce(t, op="mean")
    finally:
        dist.destroy_process_group()
