"""Which kernels a message-passing step runs, and the workspace sizes and launch counts that follow (host only, no device).

The C-ABI resolves each step's path once from its descriptor: the edge kernel (SIMT, first-generation tcgen05, the second- or
third-generation fused kernels, or the edge MLP as GEMMs over materialised edge rows) and the node level (the fused node kernels,
the second generation's node adjoints on tcgen05 with one reduction of all partials, or generic GEMMs).  The sizes and counts are
public: callers allocate workspaces by them and bench.py adds up the launches.  They are pinned here for descriptors that cover
every path.  Sizes that depend on the SM count are for 148 SMs: a B200 has 148, and without a device the library assumes 148."""
import pytest

from gnn_jet_autoencoder_b200 import _lib

FP32, BF16 = 0, 1
EUC, MINK = 0, 1
D = [32, 128, 64, 16]      # the default edge widths

# precision, B, N, H, edge widths, node widths, alpha, metric, h_ld, h_cols (0: node_in), path,
# (parameters, forward workspace, backward workspace, saved, partials, launches (forward, backward, backward on saved)).
# path: the edge kernel (simt, tc1, tc2, tc3, mat) + the node level: "fused" node kernels, "tail" (both node adjoints on tcgen05
# and one reduction of all partials) or "dense" (generic GEMMs).
TABLE = [
    # the steps of test_gpu_parity.py::test_mp_step_matches_oracle
    (FP32, 3, 30, 16, D, [16, 32], 0.2, EUC, 0, 0, "simt+fused", (15680, 23040, 227328, 0, 0, (3, 8, 8))),
    (BF16, 3, 30, 16, D, [16, 32], 0.2, EUC, 0, 0, "tc2+tail", (15680, 65280, 8762880, 65280, 8656640, (4, 8, 5))),
    (FP32, 5, 6, 4, D, [4, 4], 0.2, MINK, 0, 0, "simt+fused", (13944, 7680, 294400, 0, 0, (3, 8, 8))),
    (BF16, 5, 6, 4, D, [4, 4], 0.2, MINK, 0, 0, "tc2+tail", (13944, 42240, 8251392, 42240, 8195072, (4, 8, 5))),
    (FP32, 2, 150, 32, D, [32, 8], 0.2, EUC, 0, 0, "simt+fused", (17464, 76800, 297984, 0, 0, (3, 8, 8))),
    (BF16, 2, 150, 32, D, [32, 8], 0.2, EUC, 0, 0, "tc2+tail", (17464, 395520, 10081536, 299520, 9301248, (5, 9, 6))),
    (FP32, 3, 31, 16, D, [16, 32], 0.2, EUC, 0, 0, "simt+fused", (15680, 23808, 229120, 0, 0, (3, 8, 8))),
    (BF16, 3, 31, 16, D, [16, 32], 0.2, EUC, 0, 0, "tc2+tail", (15680, 66560, 8765696, 66560, 8656640, (4, 8, 5))),
    (FP32, 3, 32, 16, D, [16, 32], 0.2, EUC, 0, 0, "simt+fused", (15680, 24576, 230656, 0, 0, (3, 8, 8))),
    (BF16, 3, 32, 16, D, [16, 32], 0.2, EUC, 0, 0, "tc2+tail", (15680, 67584, 8767744, 67584, 8656640, (4, 8, 5))),
    (FP32, 2, 64, 8, D, [8, 8], 0.2, EUC, 0, 0, "simt+fused", (14368, 32768, 186624, 0, 0, (3, 8, 8))),
    (BF16, 2, 64, 8, D, [8, 8], 0.2, EUC, 0, 0, "tc2+tail", (14368, 112640, 8551936, 96256, 8348416, (5, 9, 6))),
    (FP32, 1, 96, 16, D, [16, 32], 0.2, EUC, 0, 0, "simt+fused", (15680, 24576, 113920, 0, 0, (3, 8, 8))),
    (BF16, 1, 96, 16, D, [16, 32], 0.2, EUC, 0, 0, "tc2+tail", (15680, 110592, 8854016, 92160, 8656640, (5, 9, 6))),
    (FP32, 1, 160, 16, D, [16, 32], 0.2, EUC, 0, 0, "simt+fused", (15680, 40960, 150784, 0, 0, (3, 8, 8))),
    (BF16, 1, 160, 16, D, [16, 32], 0.2, EUC, 0, 0, "tc2+tail", (15680, 225280, 9095936, 174080, 8665088, (5, 9, 6))),
    (FP32, 3, 30, 64, [64, 64], [64, 64], 0.2, EUC, 0, 0, "simt+dense", (24896, 69120, 1553920, 0, 0, (6, 23, 23))),
    (BF16, 3, 30, 64, [64, 64], [64, 64], 0.2, EUC, 0, 0, "tc3+dense", (24896, 135936, 8722944, 112896, 0, (8, 26, 19))),
    (FP32, 2, 33, 128, [128, 128], [128, 128], 0.2, EUC, 0, 0, "mat+dense", (98944, 2350080, 8065024, 0, 0, (9, 36, 36))),
    (BF16, 2, 33, 128, [128, 128], [128, 128], 0.2, EUC, 0, 0, "tc3+dense", (98944, 288256, 31079168, 186880, 0, (9, 27, 20))),
    (FP32, 2, 9, 256, [256, 256], [256, 256], 0.2, EUC, 0, 0, "mat+dense", (394496, 389632, 7916032, 0, 0, (9, 36, 36))),
    (BF16, 2, 9, 256, [256, 256], [256, 256], 0.2, EUC, 0, 0, "mat+dense", (394496, 389632, 7916032, 0, 0, (9, 36, 36))),
    (FP32, 7, 5, 4, [16, 16], [4, 4], 0.2, MINK, 0, 0, "simt+fused", (536, 4608, 23808, 0, 0, (3, 8, 8))),
    (BF16, 7, 5, 4, [16, 16], [4, 4], 0.2, MINK, 0, 0, "tc1+fused", (536, 4608, 23808, 0, 0, (3, 8, 8))),
    (FP32, 2, 33, 8, [16, 32, 16], [8, 16, 8], 0.2, EUC, 0, 0, "simt+fused", (1840, 8448, 32256, 0, 0, (3, 8, 8))),
    (BF16, 2, 33, 8, [16, 32, 16], [8, 16, 8], 0.2, EUC, 0, 0, "tc1+fused", (1840, 8448, 32256, 0, 0, (3, 8, 8))),
    (FP32, 4, 1, 3, [16], [3, 2], 0.2, EUC, 0, 0, "simt+fused", (196, 512, 3328, 0, 0, (3, 8, 8))),
    (BF16, 4, 1, 3, [16], [3, 2], 0.2, EUC, 0, 0, "simt+fused", (196, 512, 3328, 0, 0, (3, 8, 8))),
    (FP32, 2, 64, 6, [8, 24], [6, 5], 0.2, EUC, 0, 0, "simt+fused", (549, 16384, 47872, 0, 0, (3, 8, 8))),
    (BF16, 2, 64, 6, [8, 24], [6, 5], 0.2, EUC, 0, 0, "tc1+fused", (549, 16384, 47872, 0, 0, (3, 8, 8))),
    (FP32, 3, 10, 8, [16, 16], [180, 180], 0.2, EUC, 0, 0, "simt+dense", (37640, 25600, 1442048, 0, 0, (6, 23, 23))),
    (BF16, 3, 10, 8, [16, 16], [180, 180], 0.2, EUC, 0, 0, "tc1+dense", (37640, 25600, 1442048, 0, 0, (6, 23, 23))),
    # test_gpu_parity.py::test_mp_step_alpha_range: alpha > 1 hands the first-generation kernels' work to the SIMT kernels
    (FP32, 3, 12, 8, [32, 64, 16], [8, 6], 0.0, EUC, 0, 0, "simt+fused", (3982, 9216, 65536, 0, 0, (3, 8, 8))),
    (BF16, 3, 12, 8, [32, 64, 16], [8, 6], 0.0, EUC, 0, 0, "tc1+fused", (3982, 9216, 65536, 0, 0, (3, 8, 8))),
    (FP32, 3, 12, 8, [32, 64, 16], [8, 6], 1.0, EUC, 0, 0, "simt+fused", (3982, 9216, 65536, 0, 0, (3, 8, 8))),
    (BF16, 3, 12, 8, [32, 64, 16], [8, 6], 1.0, EUC, 0, 0, "tc1+fused", (3982, 9216, 65536, 0, 0, (3, 8, 8))),
    (FP32, 3, 12, 8, [32, 64, 16], [8, 6], 1.7, EUC, 0, 0, "simt+fused", (3982, 9216, 65536, 0, 0, (3, 8, 8))),
    (BF16, 3, 12, 8, [32, 64, 16], [8, 6], 1.7, EUC, 0, 0, "tc1+fused", (3982, 9216, 65536, 0, 0, (3, 8, 8))),
    # the training steps of bench.py's default widths, B = 4096 at N = 30 and B = 2048 at N = 150
    (FP32, 4096, 30, 16, D, [16, 32], 0.2, EUC, 0, 0, "simt+fused", (15680, 31457280, 79426816, 0, 0, (3, 8, 8))),
    (BF16, 4096, 30, 16, D, [16, 32], 0.2, EUC, 0, 0, "tc2+tail", (15680, 47216640, 115001088, 47216640, 12733696, (4, 8, 5))),
    (FP32, 4096, 30, 32, D, [32, 8], 0.2, EUC, 0, 0, "simt+fused", (17464, 31457280, 80033024, 0, 0, (3, 8, 8))),
    (BF16, 4096, 30, 32, D, [32, 8], 0.2, EUC, 0, 0, "tc2+tail", (17464, 47216640, 117701376, 47216640, 15433984, (4, 8, 5))),
    (FP32, 4096, 30, 8, D, [8, 20], 0.2, EUC, 0, 0, "simt+fused", (14476, 31457280, 79123712, 0, 0, (3, 8, 8))),
    (BF16, 4096, 30, 8, D, [8, 20], 0.2, EUC, 0, 0, "tc2+tail", (14476, 47216640, 112386304, 47216640, 10118912, (4, 8, 5))),
    (FP32, 4096, 30, 8, D, [8, 3], 0.2, EUC, 0, 0, "simt+fused", (14323, 31457280, 79123712, 0, 0, (3, 8, 8))),
    (BF16, 4096, 30, 8, D, [8, 3], 0.2, EUC, 0, 0, "tc2+tail", (14323, 47216640, 112092672, 47216640, 9825280, (4, 8, 5))),
    (FP32, 2048, 150, 16, D, [16, 32], 0.2, EUC, 0, 0, "simt+fused", (15680, 78643200, 185595136, 0, 0, (3, 8, 8))),
    (BF16, 2048, 150, 16, D, [16, 32], 0.2, EUC, 0, 0, "tc2+tail", (15680, 373585920, 779536384, 275281920, 12733696, (5, 9, 6))),
    (FP32, 2048, 150, 32, D, [32, 8], 0.2, EUC, 0, 0, "simt+fused", (17464, 78643200, 186201344, 0, 0, (3, 8, 8))),
    (BF16, 2048, 150, 32, D, [32, 8], 0.2, EUC, 0, 0, "tc2+tail", (17464, 373585920, 782902272, 275281920, 16099584, (5, 9, 6))),
    (FP32, 2048, 150, 8, D, [8, 20], 0.2, EUC, 0, 0, "simt+fused", (14476, 78643200, 185292032, 0, 0, (3, 8, 8))),
    (BF16, 2048, 150, 8, D, [8, 20], 0.2, EUC, 0, 0, "tc2+tail", (14476, 373585920, 776921600, 275281920, 10118912, (5, 9, 6))),
    # the encoder's first step (3 input columns, zero-padded) and the decoder's (20 columns, cropped)
    (FP32, 4096, 30, 16, D, [16, 32], 0.2, EUC, 3, 3, "simt+fused", (15680, 31457280, 79426816, 0, 0, (3, 8, 8))),
    (BF16, 4096, 30, 16, D, [16, 32], 0.2, EUC, 3, 3, "tc2+tail", (15680, 47216640, 115001088, 47216640, 12733696, (4, 8, 5))),
    (FP32, 4096, 30, 16, D, [16, 32], 0.2, EUC, 20, 16, "simt+fused", (15680, 31457280, 79426816, 0, 0, (3, 8, 8))),
    (BF16, 4096, 30, 16, D, [16, 32], 0.2, EUC, 20, 16, "tc2+tail", (15680, 47216640, 115001088, 47216640, 12733696, (4, 8, 5))),
    # bench.py's config-5 sweep: edge [[H, H]], node [[H]], B = 2048 (512 at H = 256)
    (FP32, 2048, 30, 64, [64, 64], [64], 0.2, EUC, 0, 0, "simt+dense", (20736, 31457280, 151529472, 0, 0, (5, 19, 19))),
    (BF16, 2048, 30, 64, [64, 64], [64], 0.2, EUC, 0, 0, "tc3+dense", (20736, 55059456, 180609536, 55059456, 0, (7, 22, 16))),
    (FP32, 2048, 30, 128, [128, 128], [128], 0.2, EUC, 0, 0, "mat+dense", (82432, 465085952, 765620736, 0, 0, (24, 158, 158))),
    (BF16, 2048, 30, 128, [128, 128], [128], 0.2, EUC, 0, 0, "tc3+dense", (82432, 102270976, 391774720, 102270976, 0, (7, 22, 16))),
    (FP32, 512, 30, 256, [256, 256], [256], 0.2, EUC, 0, 0, "mat+dense", (328704, 432995328, 749874688, 0, 0, (16, 88, 88))),
    (BF16, 512, 30, 256, [256, 256], [256], 0.2, EUC, 0, 0, "mat+dense", (328704, 432995328, 749874688, 0, 0, (16, 88, 88))),
    # the second-generation edge kernels with the projections' adjoint alone on tcgen05, and with neither node adjoint
    (FP32, 64, 30, 16, D, [16, 64], 0.2, EUC, 0, 0, "simt+dense", (16224, 614400, 7491584, 0, 0, (6, 23, 23))),
    (BF16, 64, 30, 16, D, [16, 64], 0.2, EUC, 0, 0, "tc2+fused", (16224, 768000, 10276608, 768000, 0, (4, 10, 7))),
    (FP32, 64, 30, 48, D, [16, 32], 0.2, EUC, 0, 0, "simt+fused", (18240, 491520, 5369856, 0, 0, (3, 8, 8))),
    (BF16, 64, 30, 48, D, [16, 32], 0.2, EUC, 0, 0, "tc2+fused", (18240, 768000, 11489024, 768000, 0, (4, 10, 7))),
    # an empty batch
    (FP32, 0, 30, 16, D, [16, 32], 0.2, EUC, 0, 0, "simt+fused", (15680, 0, 58624, 0, 0, (3, 8, 8))),
    (BF16, 0, 30, 16, D, [16, 32], 0.2, EUC, 0, 0, "tc2+tail", (15680, 30720, 8687872, 30720, 0, (4, 8, 5))),
]


def observed_path(lib, d, n_node_layers):
    """The path as the launch counts show it.  The SIMT and the first-generation kernels launch alike and size their workspaces
    alike, so both read as "kernel"; the table's label says which one the mode selects (bf16 with more than one edge layer:
    the first generation)."""
    fwd, bwd, bwd_saved = (lib.gj_mp_step_launches(d, b, s) for b, s in ((0, 0), (1, 0), (1, 1)))
    if lib.gj_mp_step_saved_bytes(d):      # the fused kernels keep their by-products for the backward
        if bwd - bwd_saved == 4 + n_node_layers + 1:
            return "tc3+dense"
        assert bwd - bwd_saved == 3
        j_block_sum = fwd - 4
        return "tc2+tail" if bwd_saved - j_block_sum == 5 else "tc2+fused"      # one reduction of all partials, or three
    if fwd == 3:      # projections, edge kernel, node MLP
        return "kernel+fused"
    return "kernel+dense" if fwd == n_node_layers + 4 else "mat+dense"


def row_id(row):
    prec, B, N, H, edge, node, alpha, metric, ld, cols = row[:10]
    crop = f"-ld{ld}-cols{cols}" if cols else ""
    return (f"{'bf16' if prec else 'fp32'}-B{B}-N{N}-H{H}-e{'.'.join(map(str, edge))}-n{'.'.join(map(str, node))}-a{alpha}"
            f"{'-mink' if metric else ''}{crop}")


@pytest.mark.parametrize("row", TABLE, ids=[row_id(r) for r in TABLE])
def test_step_sizes_and_launches(row):
    prec, B, N, H, edge, node, alpha, metric, ld, cols, path, values = row
    lib = _lib.load()
    d = _lib.make_desc(B, N, H, edge, node, alpha, metric, prec, h_ld=ld, h_cols=cols)
    got = (lib.gj_mp_param_count(d), lib.gj_mp_step_fwd_workspace(d), lib.gj_mp_step_bwd_workspace(d), lib.gj_mp_step_saved_bytes(d),
           lib.gj_mp_step_partials_bytes(d), tuple(lib.gj_mp_step_launches(d, b, s) for b, s in ((0, 0), (1, 0), (1, 1))))
    assert got == values
    assert observed_path(lib, d, len(node)) == path.replace("simt+", "kernel+").replace("tc1+", "kernel+")
    assert (lib.gj_mp_step_partials_bytes(d) > 0) == (path == "tc2+tail" and B > 0)


def test_table_covers_every_path():
    paths = {row[10] for row in TABLE}
    assert paths == {"simt+fused", "simt+dense", "tc1+fused", "tc1+dense", "tc2+tail", "tc2+fused", "tc3+dense", "mat+dense"}
