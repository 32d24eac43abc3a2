"""Checkpoint files written by the UNMODIFIED reference ``PartialFC`` (``partial_fc.py:71-76`` save_params / save_FC) for
``tests/test_shard_io.py``: a seeded 300 x 64 fp32 shard and its momentum, rank 0.

    python tests/golden/make_golden_shard_io.py <FedFR checkout> tests/golden/shard_io

Writes ``rank:0_softmax_weight.pt``, ``rank:0_softmax_weight_mom.pt`` (save_params) and ``FC_rank_0.pth`` (save_FC).
The stored files were written without a checkout at hand, by the statements those two methods consist of
(``torch.save(weight.data, weight_name)``, ``torch.save(weight_mom, weight_mom_name)``,
``torch.save(weight.data, prefix/FC_rank_<local_rank>.pth)``) on the same seeded CPU tensors; running this script with a
checkout rewrites them through the class itself.
"""
import os
import sys

import torch


def main(ref, out):
    sys.path.insert(0, ref)
    import partial_fc
    r = partial_fc.PartialFC.__new__(partial_fc.PartialFC)         # its ctor hard-codes CUDA (partial_fc.py:27,61,69)
    torch.nn.Module.__init__(r)
    os.makedirs(out, exist_ok=True)
    g = torch.Generator().manual_seed(4)
    r.prefix, r.rank, r.local_rank = out, 0, 0
    r.weight = torch.randn(300, 64, generator=g) * 0.01
    r.weight_mom = torch.randn(300, 64, generator=g) * 0.001
    r.weight_name = os.path.join(r.prefix, "rank:{}_softmax_weight.pt".format(r.rank))          # partial_fc.py:38-39
    r.weight_mom_name = os.path.join(r.prefix, "rank:{}_softmax_weight_mom.pt".format(r.rank))
    r.save_params()
    r.save_FC()
    print(sorted(os.listdir(out)))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
