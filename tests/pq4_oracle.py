"""Test doubles for IVF-PQ shards with 4-bit codes.

The C oracle keeps one code per byte for any ksub; the engine, the state dicts and faiss files carry
rows of M * nbits / 8 bytes in faiss bit order.  `PackedOracleIVFPQ` converts at get_state /
set_state (faiss_io.pack_codes / unpack_codes), so that oracle and engine states can be exchanged
and compared byte for byte."""
from distributed_faiss_b200 import faiss_io
from oracle import oracle as O
from tests.oracle_engine import oracle_engine_factory


class PackedOracleIVFPQ(O.OracleIVFPQ):
    def __init__(self, d, nlist, M, nbits=8, coarse_metric=O.METRIC_L2):
        super().__init__(d, nlist, M, nbits, coarse_metric=coarse_metric)
        self.nbits = int(nbits)

    def get_state(self):
        st = super().get_state()
        st["codes"] = faiss_io.pack_codes(self.codes, self.nbits)
        return st

    def set_state(self, st, recompute_tvals=True):
        st = dict(st)
        st["codes"] = faiss_io.unpack_codes(st["codes"], self.M, self.nbits)
        super().set_state(st, recompute_tvals)


def packed_oracle_engine_factory(cfg):
    """oracle_engine_factory with knnlm shards that exchange packed codes"""
    if cfg.index_builder_type == "knnlm":
        ix = PackedOracleIVFPQ(cfg.dim, int(cfg.centroids), int(cfg.extra.get("code_size", 64)),
                               int(cfg.extra.get("bits_per_vector", 8)), coarse_metric=cfg.get_metric())
        cfg.nprobe = ix.nprobe
        return ix
    return oracle_engine_factory(cfg)
