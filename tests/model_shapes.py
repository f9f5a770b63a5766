"""Model shapes beyond v0.4.0 that the library accepts, with the kernels each one must get.

Shared by test_model_shapes_host.py (the kernel choice and workspace sizes, no GPU) and test_model_shapes_gpu.py (the
kernels against the float64 oracle).  Every shape is `bench.V040` with a few hyper-parameters changed.  The tensor-core
read kernels claim d_read <= 31, d_info + d_seq <= 32, H = d_ffn / 2 <= 11, d_feat <= 16, K <= 6 and up to 12 gated
blocks (pmt_tc_supported); the SIMT kernels go to d_model 64, d_feat 32 and K 14.
"""
from dataclasses import dataclass, field

import numpy as np
import torch

import bench

V040_CNN = list(bench.V040["ref_seq_layer_strings"])


@dataclass(frozen=True)
class Shape:
    name: str
    changes: dict = field(default_factory=dict)
    reads_tc: bool = True            # the tensor-core read kernels take this shape (tf32x3 / tf32)
    cnn_tc: bool = True              # the tensor-core haplotype CNN takes it
    n_info: int = 71
    n_read_features: int = 61        # decoded width F; compressed rows of F - 49 bytes (7 packed + F - 56 quantised)
    hap_len: int = 21                # per haplotype; the model's haplotypes_length is twice this
    num_sources: int = 1
    seed: int = 0                    # build_model's seed: logits of both signs, mostly far from saturation
    bwd_reads_tc: bool = None        # the tensor-core read-path backward (tf32x3 / tf32); None: same as reads_tc
    trains: bool = True              # False: the FP32 read-path backward's shared-memory plan does not fit, pmt_backward refuses

    @property
    def bwd_tc(self) -> bool:
        return self.reads_tc if self.bwd_reads_tc is None else self.bwd_reads_tc

    @property
    def row_bytes(self) -> int:
        return self.n_read_features - 49

    @property
    def hp(self) -> dict:
        return dict(bench.V040, **self.changes, num_sources=self.num_sources)


# the corners of the tensor-core envelope (H 1, self_attention_hidden_dimension 2, is refused: pmt_build_plan)
TC_SHAPES = [
    Shape("max_corner", dict(read_layers=[31, -2], info_layers=[22], self_attention_hidden_dimension=22,
                             aggregation_layers=[-2, 16], num_artifact_clusters=6), seed=4, trains=False),       # 31 / 32 / H 11 / E 16 / K 6
    Shape("min_corner", dict(read_layers=[8, -1], info_layers=[4], self_attention_hidden_dimension=4,
                             num_self_attention_layers=1, aggregation_layers=[2], num_artifact_clusters=1,
                             ref_seq_layer_strings=V040_CNN[:-1] + ["linear/out_features=4"])),   # 8 / 8 / H 2 / E 2 / K 1
    Shape("deep_odd", dict(read_layers=[17, -3, -1], info_layers=[13, -1], self_attention_hidden_dimension=14,
                           num_self_attention_layers=12, aggregation_layers=[-1, -3, 9], num_artifact_clusters=5),
          num_sources=2),                            # 17 / 23 / H 7 / 12 blocks / E 9 / K 5
    Shape("e1", dict(aggregation_layers=[1]), seed=4),                                                # E - 1 = 0 in the head
]
# d_model 64, E 32, K 14: the SIMT kernels' limits
SIMT_SHAPES = [
    Shape("simt_limits", dict(read_layers=[24, -2], info_layers=[30], self_attention_hidden_dimension=64,
                              aggregation_layers=[-2, 32], num_artifact_clusters=14), reads_tc=False, seed=1, trains=False),
]
# one past each edge of the tensor-core envelope: the SIMT kernels run, the tensor-core forward refuses
EDGE_SHAPES = [
    Shape("d_read_32", dict(read_layers=[32, -2, -2, -2]), reads_tc=False, seed=1),
    Shape("d_info_seq_33", dict(info_layers=[23, -2, -2, -2]), reads_tc=False),
    Shape("h_12", dict(self_attention_hidden_dimension=24), reads_tc=False, seed=4, trains=False),
    Shape("e_17", dict(aggregation_layers=[-2, -2, 17]), reads_tc=False, seed=1),
    Shape("k_7", dict(num_artifact_clusters=7), reads_tc=False, seed=4),
    Shape("read_two_linears", dict(read_layers=[30, 30]), reads_tc=False),
    Shape("read_one_linear", dict(read_layers=[30]), reads_tc=False, seed=6),
]
# the info MLP's kernels: info_mlp_rows_kernel<8> (and the warp kernel) at width 32, the tile GEMM over 32, other inputs
INFO_SHAPES = [
    Shape("info_w32", dict(info_layers=[32, -1], read_layers=[22, -2]), reads_tc=False),      # d_model 64: FP32 only
    Shape("info_tile_gemm", dict(info_layers=[40, 20]), seed=1),
    Shape("n_info_9", n_info=9),
    Shape("n_info_128", n_info=128, seed=1),
]
# haplotype lengths the tensor-core CNN does not take (see pmt_build_cnn_tc_plan)
HAP_SHAPES = [
    Shape("hap_50", hap_len=25, cnn_tc=False, seed=3),    # flatten keeps 2 positions: the weight images overflow shared memory
    Shape("hap_64", hap_len=32, cnn_tc=False, seed=5),    # an odd length reaches the stride-2 pool
]
ALL_SHAPES = TC_SHAPES + SIMT_SHAPES + EDGE_SHAPES + INFO_SHAPES + HAP_SHAPES
BY_NAME = {s.name: s for s in ALL_SHAPES}


def build_model(shape: Shape, device, seed=None):
    """An ArtifactModel of this shape with every parameter moved away from its initialisation (seeded, by default with
    the shape's own seed), so that no folded term -- LayerNorm affine, ref regulariser, gate scalars, skip alphas,
    reg_weight, the rotation, the cluster parameters -- is numerically hidden."""
    from helpers import params_from_hp
    from permutect_b200.architecture.artifact_model import ArtifactModel
    hp = shape.hp
    seed = shape.seed if seed is None else seed
    torch.manual_seed(seed)
    model = ArtifactModel(params_from_hp(hp), shape.n_read_features, shape.n_info, 2 * shape.hap_len, device=torch.device("cpu"))
    if shape.num_sources > 1:
        model.reset_source_predictor(shape.num_sources)
    model.source_predictor.set_adversarial_strength(0.3)
    gen = torch.Generator().manual_seed(1000 + seed)
    rnd = lambda p: torch.randn(p.shape, generator=gen)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if p.dim() == 0:                                   # gate scalars, skip alphas, reg_weight
                p.copy_(0.1 + 0.4 * torch.rand((), generator=gen))
            elif name.endswith("norm.weight"):
                p.copy_(1.0 + 0.25 * rnd(p))
            elif name.endswith("norm.bias") or "regularizer" in name:
                p.copy_(0.2 * rnd(p))
            elif name.startswith("feature_clustering") or "rotation" in name:
                p.add_(0.3 * rnd(p))
            else:
                p.add_(0.2 * p.abs().mean() * rnd(p))
    return model.to(device)


def make_raw(shape: Shape, n_variants: int, seed: int) -> dict:
    """WGS-shaped ragged variants (synthetic.make_arrays) with this shape's info width and haplotype length, as the
    oracle's raw arrays."""
    from permutect_b200.synthetic import make_arrays, wgs_counts
    rng = np.random.default_rng(seed)
    ref, alt = wgs_counts(n_variants, rng)
    ia, fa, reads = make_arrays(ref, alt, rng, n_info=shape.n_info, hap_len=shape.hap_len, row_bytes=shape.row_bytes)
    sources = rng.integers(0, shape.num_sources, n_variants) if shape.num_sources > 1 else np.zeros(n_variants, np.int64)
    return dict(reads_u8=reads, read_indices=None, ref_counts=ia[:, 0].astype(np.int64), alt_counts=ia[:, 1].astype(np.int64),
                info=fa[:, 6:].astype(np.float32), haplotypes=ia[:, 16:], labels=ia[:, 2].astype(np.int64),
                sources=sources.astype(np.int64))


def long_set_raw(shape: Shape, sets, seed: int) -> dict:
    """Variants of the given (ref, alt) read counts (sets longer than a tile among them), this shape's widths."""
    from permutect_b200.synthetic import make_arrays
    rng = np.random.default_rng(seed)
    ref = np.array([r for r, _ in sets], np.int64)
    alt = np.array([a for _, a in sets], np.int64)
    ia, fa, reads = make_arrays(ref, alt, rng, n_info=shape.n_info, hap_len=shape.hap_len, row_bytes=shape.row_bytes)
    B = len(sets)
    sources = rng.integers(0, shape.num_sources, B) if shape.num_sources > 1 else np.zeros(B, np.int64)
    return dict(reads_u8=reads, read_indices=None, ref_counts=ref, alt_counts=alt, info=fa[:, 6:].astype(np.float32),
                haplotypes=ia[:, 16:], labels=ia[:, 2].astype(np.int64), sources=sources.astype(np.int64))
