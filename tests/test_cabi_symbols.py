"""The C-ABI library loads on a CPU-only box and exports every symbol the header declares
(no compute calls here).  Host-only entry points are exercised."""
import ctypes as C

import pytest

from b200 import _native as N
from b200 import atlas as A
from csrc_build import ensure_built


@pytest.fixture(scope="module", autouse=True)
def _built():
    ensure_built()


def test_every_declared_symbol_is_exported_and_bound():
    declared = set(N.header_functions())
    assert declared, "header parse found nothing"
    assert declared == set(N.SIGNATURES), declared ^ set(N.SIGNATURES)
    handle = C.CDLL(N.LIB_PATH)
    for name in declared:
        assert hasattr(handle, name), name
    assert N.lib().b200_version() >= 100


def test_flat_layout_matches_reference_parameter_counts():
    lib = N.lib()
    m = A.make_desc(**A.MAPPING_DESC)
    a = A.make_desc(**A.ATLAS_DESC)
    mw, mb, mt = A.mlp_layout(m)
    aw, ab, at = A.mlp_layout(a)
    # unpadded counts printed by IMLP.__init__ in the reference: 264706 / 416379 (SURVEY §8)
    assert sum(k * n + n for k, n in A.layer_dims(m)) == 264706
    assert sum(k * n + n for k, n in A.layer_dims(a)) == 416379
    assert mt == 264708 and at == 416380 and lib.b200_atlas_param_floats() == mt + at
    assert all(o % 4 == 0 for o in mw + mb + aw + ab)
    assert A.layer_dims(a)[4] == (296, 256) and A.layer_dims(a)[7] == (296, 3)


def test_invalid_descriptor_is_rejected_with_message():
    bad = N.MlpDesc(3, 2, 256, 1, 0, 0, 1, 0)          # a 1-layer network is not an IMLP
    assert N.lib().b200_mlp_layout(C.byref(bad), None, None) == -1
    assert b"invalid" in N.lib().b200_last_error()


def test_tc_architecture_accepts_exactly_the_stage1_shapes():
    """b200_mlp_tc_architecture: 1 for the mapping (6 or 4 layers), 2 atlas, 3 alpha; a shape one attribute away from
    one of them has no tensor-core kernels (0); an invalid descriptor is -1."""
    def arch(in_dim, out_dim, hidden, layers, pe, skips):
        d = N.MlpDesc(in_dim, out_dim, hidden, layers, pe, sum(1 << l for l in skips), 1, 0)
        return N.lib().b200_mlp_tc_architecture(C.byref(d))
    mapping6, mapping4 = (3, 2, 256, 6, 0, ()), (3, 2, 256, 4, 0, ())
    atlas, alpha = (2, 3, 256, 8, 10, (4, 7)), (3, 1, 256, 8, 5, ())
    assert [arch(*s) for s in (mapping6, mapping4, atlas, alpha)] == [1, 1, 2, 3]
    near_misses = [
        (3, 2, 256, 5, 0, ()), (3, 2, 256, 7, 0, ()),                 # layers
        (2, 3, 256, 7, 10, (4,)), (2, 3, 256, 9, 10, (4, 7)), (3, 1, 256, 7, 5, ()), (3, 1, 256, 9, 5, ()),
        (3, 2, 128, 6, 0, ()), (3, 2, 128, 4, 0, ()), (2, 3, 128, 8, 10, (4, 7)), (3, 1, 128, 8, 5, ()),   # hidden
        (2, 3, 256, 8, 9, (4, 7)), (3, 1, 256, 8, 4, ()), (3, 2, 256, 6, 4, ()),                          # pe
        (2, 2, 256, 6, 0, ()), (3, 3, 256, 6, 0, ()), (3, 3, 256, 8, 10, (4, 7)), (2, 2, 256, 8, 10, (4, 7)),
        (2, 1, 256, 8, 5, ()), (3, 2, 256, 8, 5, ()),                                                    # widths
        (2, 3, 256, 8, 10, (4,)), (2, 3, 256, 8, 10, (7,)),           # atlas with one of its two skips
        (2, 3, 256, 8, 10, (2, 4, 7)), (3, 1, 256, 8, 5, (4,)),       # an extra skip
        (3, 2, 256, 6, 0, (3,)), (3, 2, 256, 4, 0, (2,)),             # a mapping with a skip
    ]
    assert [arch(*s) for s in near_misses] == [0] * len(near_misses)
    assert arch(3, 2, 256, 1, 0, ()) == -1


def test_workspace_sizes_are_positive_and_monotone():
    lib = N.lib()
    small = N.AtlasConfig(1000, 1, N.PREC_FP32, 768, 0.8, 1, 100, 5000, 1000, 1, 5, 500)
    big = N.AtlasConfig(10000, 1, N.PREC_FP32, 768, 0.8, 1, 100, 5000, 1000, 1, 5, 500)
    a, b = lib.b200_atlas_workspace_bytes(C.byref(small)), lib.b200_atlas_workspace_bytes(C.byref(big))
    assert 0 < a < b
    assert lib.b200_render_workspace_bytes(1000) > 0
    assert lib.b200_render_workspace_bytes(0) == -1
    # the plan takes at most 16384 samples per iteration; one more is refused with a message, not truncated
    edge = N.AtlasConfig(16384, 1, N.PREC_TC, 768, 0.8, 1, 100, 5000, 1000, 1, 5, 500)
    over = N.AtlasConfig(16385, 1, N.PREC_TC, 768, 0.8, 1, 100, 5000, 1000, 1, 5, 500)
    assert lib.b200_atlas_workspace_bytes(C.byref(edge)) > b
    assert lib.b200_atlas_workspace_bytes(C.byref(over)) == -1 and b"16384" in lib.b200_last_error()


def test_frame_ranges_partition_the_video():
    for T in (80, 7, 16):
        for world in (1, 2, 4, 8):
            spans = [A.frame_range(r, world, T) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == T
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            assert max(b - a for a, b in spans) - min(b - a for a, b in spans) <= 1


def _conv_desc(n, cin, h, w, cout, kh, kw, stride=1, pad=(0, 0), pad_mode=0, upsample=1, up_mode=0):
    return N.ConvDesc(n, cin, h, w, cin, 0, cout, kh, kw, stride, pad[0], pad[1], pad_mode, upsample, cout, 0, 0, 1.0, 0, 0,
                      up_mode)


def test_conv_tma_geometry_host_side():
    """Workspace / weight-image sizes of the TMA convolution are closed-form functions of the descriptor
    (conv_tma.cu tma_geometry): fp16 NHWC repack with channels padded to 64, padding / upsampling / stride-2
    phases materialised; images = cout tiles x chunks x n_tile rows x 128 B."""
    lib = N.lib()
    # 3x3, pad 1, 128 -> 128 at 24x40: HP=26, WP=42, Cp=128; chunks = 3*3*2, n_tile = 128
    d = _conv_desc(1, 128, 24, 40, 128, 3, 3, pad=(1, 1))
    assert lib.b200_conv_tma_workspace_bytes(C.byref(d)) == 26 * 42 * 128 * 2 + 256
    assert lib.b200_conv_tma_weight_image_bytes(C.byref(d)) == 18 * 128 * 128
    # stride 2 (4 pixel phases): HP2 = ceil(32/2), WP2 = ceil(46/2), Cp = 64; 9 chunks, n_tile = 64
    d = _conv_desc(1, 32, 30, 44, 64, 3, 3, stride=2, pad=(1, 1), pad_mode=1)
    assert lib.b200_conv_tma_workspace_bytes(C.byref(d)) == 4 * 16 * 23 * 64 * 2 + 256
    assert lib.b200_conv_tma_weight_image_bytes(C.byref(d)) == 9 * 64 * 128
    # narrow input, 7x7: x taps folded into the channels (8 per tap): packed width = OW, one chunk per filter row
    d = _conv_desc(2, 6, 33, 47, 32, 7, 7, pad=(3, 3), pad_mode=1)
    assert lib.b200_conv_tma_workspace_bytes(C.byref(d)) == 2 * 39 * 47 * 64 * 2 + 256
    assert lib.b200_conv_tma_weight_image_bytes(C.byref(d)) == 7 * 32 * 128
    # Cout 576 -> 3 cout tiles of 192; x2 nearest upsampling doubles the repacked extent
    d = _conv_desc(1, 256, 16, 24, 576, 1, 1)
    assert lib.b200_conv_tma_weight_image_bytes(C.byref(d)) == 3 * 4 * 192 * 128
    d = _conv_desc(1, 64, 20, 28, 32, 3, 3, pad=(1, 1), pad_mode=1, upsample=2)
    assert lib.b200_conv_tma_workspace_bytes(C.byref(d)) == 42 * 58 * 64 * 2 + 256
    # invalid descriptors are refused on the host
    for bad in (_conv_desc(1, 8, 8, 8, 8, 3, 3, stride=3), _conv_desc(1, 8, 8, 8, 8, 3, 3, pad=(9, 9), pad_mode=1),
                _conv_desc(1, 8, 8, 8, 8, 3, 3, upsample=1, up_mode=1), _conv_desc(0, 8, 8, 8, 8, 3, 3)):
        assert lib.b200_conv_tma_workspace_bytes(C.byref(bad)) == -1
    assert lib.b200_corr_build_tc_workspace_bytes(256, 135, 240) > 2 * 135 * 240 * 256 * 2
    assert lib.b200_corr_build_tc_workspace_bytes(256, 4, 240) == -1
    assert lib.b200_corr_pyramid_floats(16, 24) == 384 * (384 + 96 + 24 + 6)


def test_seg_entry_points_validate_their_arguments():
    """Host-side validation of the segmentation entry points (no GPU work): sizes, layouts, loud errors."""
    import ctypes as C
    from b200 import seg as SG
    lib = N.lib()
    d = SG.seg_descs(SG.SEG_DEFAULTS)
    cfg = N.SegConfig(10000, 1, N.PREC_FP32, 768, 0.8, 1.0, 100.0, 5000.0, 1000.0, 1.0, 5.0, 50.0, 500.0, 4900.0, 1000.0, 2000.0,
                      d["mapping1"], d["mapping2"], d["alpha"], d["atlas"])
    offs = (C.c_int64 * 4)()
    total = lib.b200_seg_param_floats(C.byref(cfg), offs)
    assert list(offs) == sorted(offs) and offs[0] == 0 and 1217152 <= total <= 1217152 + 64          # 264706 + 133122 + 402945 + 416379 parameters, each tensor padded to 4 floats
    assert [lib.b200_mlp_tc_architecture(C.byref(d[k])) for k in ("mapping1", "mapping2", "alpha", "atlas")] == [1, 1, 3, 2]
    assert lib.b200_seg_workspace_bytes(C.byref(cfg)) > 0 and lib.b200_seg_render_workspace_bytes(C.byref(cfg), 65536) > 0
    cfg.batch = 0
    assert lib.b200_seg_workspace_bytes(C.byref(cfg)) == -1 and b"samples_batch" in lib.b200_last_error()
    cfg.batch, cfg.precision = 64, 7
    assert lib.b200_seg_workspace_bytes(C.byref(cfg)) == -1 and b"precision" in lib.b200_last_error()
    cfg.precision = N.PREC_FP32
    cfg.alpha.output_dim = 2
    assert lib.b200_seg_workspace_bytes(C.byref(cfg)) == -1 and b"alpha network" in lib.b200_last_error()
    assert lib.b200_mlp_pretrain_workspace_bytes(C.byref(d["atlas"]), 10000) == -1      # pre-training is for 3 -> 2 networks
    assert lib.b200_eval_maps_workspace_bytes(C.byref(d["mapping1"]), 432 * 768) > 0
