"""Python mirror of ``plan_gemm`` (csrc/gemm.cu): the tile width, K split and partial-buffer pitch that ``hicgat_gemm_tf32_tn``
picks for a GEMM, and the branches a plan takes.  The GEMM tests use it to choose shapes that reach every branch and to know
where the split-K boundaries fall; ``test_gemm_plan_host.py`` pins it to the library's workspace size."""
from __future__ import annotations

from dataclasses import dataclass

BM, BK, MAIN_BLOCKS_MAX = 128, 32, 16


@dataclass(frozen=True)
class Plan:
    m: int
    n: int
    k: int
    kparts: int
    wide: bool
    ksplit: int
    kb_per_split: int
    kblocks: int
    ldp: int
    capped: bool  # kparts 3 and the tile rule asked for more than 16 main k-blocks per split: the cap set the split count

    @property
    def bn(self) -> int:
        return 256 if self.wide else 128

    @property
    def workspace_bytes(self) -> int:
        return self.ksplit * self.m * self.ldp * 4 if self.ksplit > 1 else 0

    def split_ranges(self):
        """``[kb0, kb1)`` k-block range of every split, in split order."""
        return [(z * self.kb_per_split, min((z + 1) * self.kb_per_split, self.kblocks)) for z in range(self.ksplit)]

    @property
    def last_short(self) -> bool:
        return self.ksplit > 1 and self.kblocks % self.kb_per_split != 0

    @property
    def main_blocks_per_acc(self) -> int:
        """Most main (hi.hi, or for kparts 1 all) k-blocks one accumulator takes."""
        return self.kb_per_split // 3 if self.kparts == 3 else self.kb_per_split

    def branches(self) -> set:
        b = {"wide" if self.wide else "narrow", f"kparts={self.kparts}", "ksplit=1" if self.ksplit == 1 else "ksplit>1"}
        if self.ksplit > 1:
            b.add("split count by cap" if self.capped else "split count by tiles")
        if self.last_short:
            b.add("last split short")
        if self.m < BM:
            b.add("m<128")
        elif self.m % BM in (1, 33, 127):
            b.add(f"m%128={self.m % BM}")
        if self.n % 32:
            b.add("n%32!=0")
        if self.wide and 0 < self.n % 256 <= 128:
            b.add("wide n%256 in (0,128]")
        if self.n % 4:
            b.add("n%4!=0")
        return b


ALL_BRANCHES = {"narrow", "wide", "kparts=1", "kparts=3", "ksplit=1", "ksplit>1", "split count by cap", "split count by tiles",
                "last split short", "m<128", "m%128=1", "m%128=33", "m%128=127", "n%32!=0", "wide n%256 in (0,128]", "n%4!=0"}


def plan_gemm(m: int, n: int, k: int, kparts: int) -> Plan:
    kblocks = (k + BK - 1) // BK
    tm = (m + BM - 1) // BM
    t128 = tm * ((n + 127) // 128)
    wide = n > 128 and t128 >= 296
    tiles = tm * ((n + 255) // 256) if wide else t128
    ks = 1
    if tiles < 148:
        ks = min(max(148 // tiles, 1), max(kblocks // 16, 1))
    kbps = (kblocks + ks - 1) // ks
    capped = False
    if kparts == 3:
        kbps = (kbps + 2) // 3 * 3
        if kbps > 3 * MAIN_BLOCKS_MAX:
            kbps, capped = 3 * MAIN_BLOCKS_MAX, True
    ksplit = (kblocks + kbps - 1) // kbps
    return Plan(m, n, k, kparts, wide, ksplit, kbps, kblocks, (n + 3) // 4 * 4, capped)


def kpad(k: int) -> int:
    return (k + BK - 1) // BK * BK


def linear_gemms(rows: int, nin: int, nout: int):
    """``(name, m, n, k')`` of the three 3xTF32 GEMMs of ``Linear(nin, nout)`` on ``rows`` rows (ops._Linear3xTF32): forward
    ``x . W^T``, dx ``dy . W`` (reduction over the output features), dW ``dy^T . x`` (reduction over the rows)."""
    return [("fwd", rows, nout, 3 * kpad(nin)), ("dx", rows, nin, 3 * kpad(nout)), ("dW", nout, nin, 3 * kpad(rows))]


def production_linears():
    """``(layer, nin, nout)`` of every Linear in the three models (models.py) and of the GATConv projection for every compiled
    (heads, channels) pair (layers.GAT_SHAPES)."""
    from hic_gnn_b200 import layers

    out = [("Net.conv.lin_l/lin_r", 512, 512), ("densea/align_densea", 512, 256), ("dense1", 256, 128), ("dense1 (v2)", 256, 64),
           ("dense2", 128, 64), ("dense3", 64, 3), ("dense2 (v2)", 64, 3)]
    out += [(f"GATConv H={h} C={c}", 512, h * c) for h, c in layers.GAT_SHAPES]
    return out


ROWS = (4096, 9970, 49850)
