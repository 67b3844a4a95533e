"""Host and device forms of every C ABI pair share one argument check: called with null handles, both return
ILSM_ERR_INVALID_ARG without a GPU (the check runs before any CUDA call), and their error texts differ only by the
entry point's name."""
import pytest

INVALID_ARG = -1

# pair -> (host call, device call), every handle null
PAIRS = {
    "map_build": (lambda L: L.ilsm_map_build(None, None, 0, 16, 0.0),
                  lambda L: L.ilsm_map_build_dev(None, None, 0, 16, 0.0)),
    "knn": (lambda L: L.ilsm_knn(None, None, 0, 16, 5, 0.0, None, None),
            lambda L: L.ilsm_knn_dev(None, None, 0, 16, 5, 0.0, None, None)),
    "register": (lambda L: L.ilsm_register(None, None, None, None, 0, None, 0, 16, None, None, None, None),
                 lambda L: L.ilsm_register_dev(None, None, None, None, 0, None, 0, 16, None, None, None)),
    "associate": (lambda L: L.ilsm_associate(None, None, None, None, 0, None, 0, 16, None, None, None, None, None, None),
                  lambda L: L.ilsm_associate_dev(None, None, None, None, 0, None, 0, 16, None, None)),
    "register_frame": (lambda L: L.ilsm_register_frame(None, None, None, None, 0, 16, 0.0, 0.2, 0.4, None, None, None, None, None),
                       lambda L: L.ilsm_register_frame_dev(None, None, None, None, 0, 16, 0.0, 0.2, 0.4, None, None)),
    "project": (lambda L: L.ilsm_project(None, None, 4, 4, 16, None, None, None),
                lambda L: L.ilsm_project_dev(None, None, 4, 4, 16, None, None, None)),
    "pc2_pack": (lambda L: L.ilsm_pc2_pack(None, None, 0, None, None),
                 lambda L: L.ilsm_pc2_pack_dev(None, None, 0, None, None)),
    "pc2_unpack": (lambda L: L.ilsm_pc2_unpack(None, None, 0, None, None),
                   lambda L: L.ilsm_pc2_unpack_dev(None, None, 0, None, None)),
    "eval_normal_eq": (lambda L: L.ilsm_eval_normal_eq(None, None, None, 0.1, None, None, None),
                       lambda L: L.ilsm_eval_normal_eq_dev(None, None, 0.1, None)),
    "solve": (lambda L: L.ilsm_solve(None, None, None, 4, 0.1, None),
              lambda L: L.ilsm_solve_dev(None, None, 4, 0.1)),
    "sc_add": (lambda L: L.ilsm_sc_add(None, None, 0),
               lambda L: L.ilsm_sc_add_dev(None, None, 0)),
    "sc_query_topk": (lambda L: L.ilsm_sc_query_topk(None, None, -1, 0, 5, None, None, None),
                      lambda L: L.ilsm_sc_query_topk_dev(None, None, -1, 0, 5, None, None, None)),
    "sc_query_topk_batch": (lambda L: L.ilsm_sc_query_topk_batch(None, None, 1, -1, 0, 5, None, None, None),
                            lambda L: L.ilsm_sc_query_topk_batch_dev(None, None, 1, -1, 0, 5, None)),
    "sc_query_topk_sharded": (lambda L: L.ilsm_sc_query_topk_sharded(None, None, 1, -1, 0, 5, None, None, None),
                              lambda L: L.ilsm_sc_query_topk_sharded_dev(None, None, 1, -1, 0, 5, None)),
    "icp_align_batch": (lambda L: L.ilsm_icp_align_batch(None, None, 1, None, None, 16, None, None, None),
                        lambda L: L.ilsm_icp_align_batch_dev(None, None, 1, None, None, 16, None, None, None)),
}


def _status(lib, call):
    rc = call(lib)
    who, _, rest = lib.ilsm_last_error().decode().partition(": ")
    return rc, who, rest


@pytest.mark.parametrize("pair", sorted(PAIRS))
def test_pair_forms_share_their_check(ilsm, pair):
    lib = ilsm.load_library()
    host, dev = PAIRS[pair]
    rc_h, who_h, msg_h = _status(lib, host)
    rc_d, who_d, msg_d = _status(lib, dev)
    assert rc_h == rc_d == INVALID_ARG, (pair, rc_h, rc_d)
    assert who_d == who_h + "_dev", (pair, who_h, who_d)
    assert msg_h and msg_h == msg_d, (pair, msg_h, msg_d)


def test_pair_build_check_without_maps(ilsm):
    """ilsm_map_build_pair_dev applies the check of ilsm_map_build to each of its two maps."""
    lib = ilsm.load_library()
    assert lib.ilsm_map_build_pair_dev(None, None, 0, None, None, 0, 16, 0.0) == INVALID_ARG
    assert lib.ilsm_last_error() == b"map_build_pair_dev: null argument"
