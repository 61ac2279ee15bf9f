"""CPU suite: the host-side data model (decomposition, compute tiles, BC / ghost-exchange /
restriction / interpolation block lists, level table, send/recv tables) is bit-identical to the
reference's for 1, 2, 4, 8 and 9 ranks.  The library runs in layout-only mode (no device)."""
import pytest

import hpgmg_b200.api as api
import oracle_bindings as ob

DECOMPS = ["5 8 x1", "5 8 x2", "5 8 x4", "5 8 x8", "4 1 x1", "6 8 x1", "6 8 x8", "4 3 x9"]


def our_summary(layout_lib, log2, bpr, ranks, rank):
    H = api.Hierarchy(log2, bpr, my_rank=rank, num_ranks=ranks, build_operator=False, library=None)
    H.L.MGBuild(H.mg, H.level_h, 0.0, 1.0, 1)     # layout-only: builds levels + lists, skips the operator rebuild
    H.built = True
    out = [ob.level_list_summary(H.level(l)) for l in range(H.num_levels)]
    active = [H.level(l).contents.active for l in range(H.num_levels)]
    H.close()
    return out, active


@pytest.mark.parametrize("key", DECOMPS)
def test_lists_equal_reference_goldens(layout_lib, key):
    cfg, x = key.rsplit(" x", 1)
    log2, bpr = map(int, cfg.split())
    ranks = int(x)
    gold = ob.goldens()["decompositions"][key]
    for r in range(ranks):
        ours, active = our_summary(layout_lib, log2, bpr, ranks, r)
        assert len(ours) == len(gold[r]), "number of levels"
        for l, (a, b) in enumerate(zip(ours, gold[r])):
            assert a == b, f"{key} rank {r} level {l}: {[k for k in a if a[k] != b[k]]}"
        # a rank is active on a level iff it owns boxes there or below (mg.c:985-986)
        owns = [lv["num_my_boxes"] > 0 for lv in ours]
        assert active == [1 if any(owns[l:]) else 0 for l in range(len(owns))] or active[0] == 1


@pytest.mark.parametrize("log2,bpr,ranks,bc", [(5, 8, 1, 1), (4, 8, 2, 1), (4, 8, 4, 1), (4, 8, 8, 1), (4, 2, 1, 1),
                                               (5, 8, 1, 0), (4, 1, 1, 0), (4, 8, 2, 0), (4, 27, 1, 0), (4, 8, 8, 0)])
def test_lists_equal_live_reference_entry_by_entry(layout_lib, log2, bpr, ranks, bc):
    """Not just digests: every blockCopy_type of every list, field by field, against the reference
    library called in this process where the reference is built, and with the pins of tests/golden/pins.json everywhere.
    bc 1: Dirichlet, 0: periodic (wrap-around neighbours, level.c:559-563, 757-761; no BC blocks, level.c:371; the
    driver's minCoarseDim 2, hpgmg-fv.c:278)."""
    for r in range(ranks):
        H = api.Hierarchy(log2, bpr, my_rank=r, num_ranks=ranks, build_operator=False, bc=bc)
        H.L.MGBuild(H.mg, H.level_h, 0.0, 1.0, 1 if bc else 2)
        H.built = True
        R = None
        if ob.have_ref():
            R = ob.RefHierarchy(log2, bpr, my_rank=r, num_ranks=ranks, build_operator=False, bc=bc)
            with ob.quiet():
                R.L.MGBuild(R.mg, R.level_h, 0.0, 1.0, 1 if bc else 2)
            R.built = True
        key = f"lists {log2} {bpr} x{ranks} rank {r} bc {bc}"
        ob.pin(f"{key}: levels", H.num_levels, R.num_levels if R else None)
        for l in range(H.num_levels):
            ob.pin(f"{key}: level {l}", repr(level_entries(H.level(l).contents)), repr(level_entries(R.level(l).contents)) if R else None)
            if l > 0:                        # level 0's h is set by the operator setup, which this test skips
                ob.pin(f"{key}: level {l} h", H.level(l).contents.h, R.level(l).contents.h if R else None)
        if R is None:
            H.close()
            continue
        assert H.num_levels == R.num_levels
        for l in range(H.num_levels):
            a, b = H.level(l).contents, R.level(l).contents
            assert (a.box_dim, a.boxes_in.i, a.num_my_boxes, a.num_ranks, a.box_jStride, a.box_volume, a.tag) == \
                   (b.box_dim, b.boxes_in.i, b.num_my_boxes, b.num_ranks, b.box_jStride, b.box_volume, b.tag)
            assert a.h == b.h or l == 0
            assert api.block_list(a.my_blocks, a.num_my_blocks) == api.block_list(b.my_blocks, b.num_my_blocks)
            for s in range(3):
                assert api.block_list(a.boundary_condition.blocks[s], a.boundary_condition.num_blocks[s]) == \
                       api.block_list(b.boundary_condition.blocks[s], b.boundary_condition.num_blocks[s]), (l, "bc", s)
                for p in range(3):
                    assert api.block_list(a.exchange_ghosts[s].blocks[p], a.exchange_ghosts[s].num_blocks[p]) == \
                           api.block_list(b.exchange_ghosts[s].blocks[p], b.exchange_ghosts[s].num_blocks[p]), (l, "exchange", s, p)
            for t in range(4):
                for p in range(3):
                    assert api.block_list(a.restriction[t].blocks[p], a.restriction[t].num_blocks[p]) == \
                           api.block_list(b.restriction[t].blocks[p], b.restriction[t].num_blocks[p]), (l, "restriction", t, p)
            for p in range(3):
                assert api.block_list(a.interpolation.blocks[p], a.interpolation.num_blocks[p]) == \
                       api.block_list(b.interpolation.blocks[p], b.interpolation.num_blocks[p]), (l, "interpolation", p)
            for b_ in range(a.num_my_boxes):
                ba, bb = a.my_boxes[b_], b.my_boxes[b_]
                assert (ba.global_box_id, ba.low.i, ba.low.j, ba.low.k, ba.dim, ba.ghosts, ba.jStride, ba.kStride, ba.volume) == \
                       (bb.global_box_id, bb.low.i, bb.low.j, bb.low.k, bb.dim, bb.ghosts, bb.jStride, bb.kStride, bb.volume)
        H.close()


def level_entries(a):
    """Every entry the test above compares with the reference, of one level."""
    out = [(a.box_dim, a.boxes_in.i, a.num_my_boxes, a.num_ranks, a.box_jStride, a.box_volume, a.tag),
           api.block_list(a.my_blocks, a.num_my_blocks)]
    for s in range(3):
        out.append(api.block_list(a.boundary_condition.blocks[s], a.boundary_condition.num_blocks[s]))
        out += [api.block_list(a.exchange_ghosts[s].blocks[p], a.exchange_ghosts[s].num_blocks[p]) for p in range(3)]
    for t in range(4):
        out += [api.block_list(a.restriction[t].blocks[p], a.restriction[t].num_blocks[p]) for p in range(3)]
    out += [api.block_list(a.interpolation.blocks[p], a.interpolation.num_blocks[p]) for p in range(3)]
    for b_ in range(a.num_my_boxes):
        ba = a.my_boxes[b_]
        out.append((ba.global_box_id, ba.low.i, ba.low.j, ba.low.k, ba.dim, ba.ghosts, ba.jStride, ba.kStride, ba.volume))
    return out


def test_survey_appendix_e_counts(layout_lib):
    """`hpgmg-fv 7 8` on one rank: tiles | local exchange BOX/STAR/NO_CORNERS | BC blocks (SURVEY.md appendix E)."""
    H = api.Hierarchy(7, 8, build_operator=False)
    H.L.MGBuild(H.mg, H.level_h, 0.0, 1.0, 1)
    H.built = True
    want = [(256, 128, 8, 2048, (784, 640, 776), (1104, 640, 1048), 9), (128, 64, 8, 512, (272, 192, 264), (464, 192, 408), 9),
            (64, 32, 8, 128, (112, 64, 104), (240, 64, 184), 9), (32, 16, 8, 32, (56, 24, 48), (152, 24, 96), 9),
            (16, 8, 8, 8, (56, 24, 48), (152, 24, 96), 9), (8, 8, 1, 1, (0, 0, 0), (26, 6, 18), 9),
            (4, 4, 1, 1, (0, 0, 0), (26, 6, 18), 9), (2, 2, 1, 1, (0, 0, 0), (26, 6, 18), 17)]
    assert H.num_levels == 8
    for l, w in enumerate(want):
        Lv = H.level(l).contents
        got = (Lv.dim.i, Lv.box_dim, Lv.num_my_boxes, Lv.num_my_blocks,
               tuple(Lv.exchange_ghosts[s].num_blocks[1] for s in range(3)),
               tuple(Lv.boundary_condition.num_blocks[s] for s in range(3)), Lv.numVectors)
        assert got == w, (l, got, w)
    H.close()


def test_problem_size_rule():
    """hpgmg-fv.c:184-197: largest cube of boxes <= target whose side has an odd part <= 11."""
    assert api.problem_size(7, 8, 1) == (128, 2)
    assert api.problem_size(7, 8, 2) == (128, 2)      # 16 boxes -> still 2^3
    assert api.problem_size(7, 8, 4) == (128, 3)      # 32 boxes -> 3^3 (384^3)
    assert api.problem_size(7, 8, 8) == (128, 4)
    assert api.problem_size(6, 1, 1) == (64, 1)
    assert api.problem_size(8, 8, 8) == (256, 4)
