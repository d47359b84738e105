"""INTEGRATION.md option 2: the reference's own predict loop with `PredictDataset` swapped for ours.

  * our PredictDataset('.pd') through DataLoader(batch_size=1000, shuffle=False, num_workers=0 / 4) collates to the 4-tuple
    PileupModel/predict.py:45-49 unpacks (tuple[str], LongTensor[N], LongTensor[N], IntTensor[N,33,18]) with the reference's
    batch boundaries;
  * the predict loop (restated in oracle/s2_restate.py, pinned to the reference Python by tests/test_oracle_pinning.py) over
    the `.pd.bin` path predict.py:215 lists, resolved through the `.pd` text, with our PredictDataset and a stub model
    returning the golden probabilities: the VCF is byte-equal to the golden file the all-reference run produced.
"""
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN


@pytest.fixture()
def pd_dir(tmp_path, small_case):
    from nanosnp_b200.postprocess import write_pd
    d = tmp_path / "out"
    (d / "predict_data").mkdir(parents=True); (d / "bin_predict_data").mkdir()
    write_pd(str(d / "predict_data" / "ctg1.pd"), "ctg1", small_case["site_pos"], small_case["ref"], small_case["windows"])
    (d / "bin_predict_data" / "ctg1.pd.bin").write_bytes(b"")          # what predict.py:215 lists; HDF5 needs PyTables (absent)
    return d


@pytest.mark.parametrize("workers", [0, 4])
def test_dataset_collates_like_the_reference(pd_dir, small_case, workers):
    import torch
    from torch.utils.data import DataLoader
    from nanosnp_b200.dataset import PredictDataset
    ds = PredictDataset(str(pd_dir / "bin_predict_data" / "ctg1.pd.bin"))
    n = len(small_case["site_pos"])
    assert len(ds) == n
    seen = 0
    for batch in DataLoader(ds, batch_size=1000, shuffle=False, num_workers=workers):        # predict.py:43
        names, pos, refb, x = batch                                                            # predict.py:45
        m = len(names)
        assert m == min(1000, n - seen) and all(isinstance(s, str) and s == "ctg1" for s in names)
        assert pos.dtype == torch.int64 and refb.dtype == torch.int64 and tuple(pos.shape) == (m,) and tuple(refb.shape) == (m,)
        assert x.dtype == torch.int32 and tuple(x.shape) == (m, 33, 18)
        assert np.array_equal(pos.numpy(), small_case["site_pos"][seen:seen + m])
        assert np.array_equal(refb.numpy(), small_case["site_refbase"][seen:seen + m])
        assert np.array_equal(x.numpy(), small_case["windows"][seen:seen + m])
        assert x.type(torch.FloatTensor).dtype == torch.float32                               # predict.py:49
        seen += m
    assert seen == n


def test_reference_predict_loop_with_our_dataset(pd_dir, monkeypatch):
    import torch
    from torch.utils.data import DataLoader
    from nanosnp_b200.dataset import PredictDataset
    from oracle.s2_restate import vcf_header, vcf_records
    monkeypatch.setitem(sys.modules, "tables", None)            # our PredictDataset must take its no-PyTables route
    z = np.load(GOLDEN / "s2_small.npz")
    text = vcf_header((GOLDEN / "s2_small.fai").read_text().splitlines())           # predict.py:13-27
    k = 0
    paths = [str(pd_dir / "bin_predict_data" / f) for f in os.listdir(pd_dir / "bin_predict_data") if f.endswith(".bin")]   # predict.py:215
    for path in paths:
        for names, pos, refb, x in DataLoader(PredictDataset(path), batch_size=1000, shuffle=False):       # predict.py:43-45
            x = x.type(torch.FloatTensor)                                                               # predict.py:49
            n = x.shape[0]
            assert x.dtype == torch.float32 and tuple(x.shape[1:]) == (33, 18)
            text += vcf_records(names, pos.numpy(), refb.numpy(), x.numpy(), z["gt"][k:k + n], z["zy"][k:k + n])
            k += n
    assert k == len(z["gt"])
    assert text.encode() == (GOLDEN / "s2_small.vcf").read_bytes()
