"""Matching accuracy and average registration error, the two numbers of the reference's `EvaluateMetrics`
widget (`_calculate_metrics`, reference _dock_widget.py:1030-1080).  SURVEY §8(f) row 3.

The three `cdist` + `linear_sum_assignment` pairs run on the GPU (pm_cdist + the exact assignment kernel of
the registration path); the dictionary bookkeeping on a handful of keypoints stays in Python as in the reference.

Without keypoints, two label volumes (e.g. the fixed segmentation and the moving one warped into its grid by
`transform_image`) are compared voxel by voxel: `label_contingency` builds their overlap table in one streaming pass
(pm_label_overlap), `match_labels` scores it as foreground Dice / Jaccard and as instance matching at IoU thresholds
(true / false positives, precision, recall, F1), the ids-free measure segmentation tools report.  DESIGN §8 row 7.
"""
import numpy as np

from . import device as D
from .utils.labels import _check_label_volume

__all__ = ["assign_by_distance", "calculate_metrics", "label_contingency", "match_labels"]

LAP_MAX_COLUMNS = 24576          # the assignment kernel's limit (pm_lap_solve refuses wider matrices)


def _check_pair(labels_a, labels_b):
    a, b = _check_label_volume(labels_a, "labels_a"), _check_label_volume(labels_b, "labels_b")
    if a.shape != b.shape:
        raise ValueError("label volumes differ in shape: %s and %s" % (a.shape, b.shape))
    return a, b


def _pow2(n):
    return 1 << max(int(n) - 1, 0).bit_length()


def _initial_capacity(max_a, max_b, n_vox):
    """Hash-table slots of the first table pass.  A segmentation pair has about two pairs per instance (its partner and
    the background): keep the table at most half full for twice that.  Sparse ids (up to 2^31 - 1) make that bound
    loose: never start above two slots per voxel or 2^24 slots (512 MB of table and output); an overflow reruns with
    more."""
    return _pow2(max(min(4 * (max_a + max_b), 2 * n_vox, 1 << 24), 1024))


def _contingency(a, b):
    """The table of two checked host volumes: (ids_a, ids_b, counts) int64 numpy arrays sorted by (a, b).
    Host synchronisations: 5 (the upload of each volume from pageable memory, the largest ids, the pair count, the
    result copy), plus 1 per overflow rerun."""
    torch = D._torch()
    ta, tb = D.to_device_volume(a), D.to_device_volume(b)
    mx = torch.zeros(2, dtype=torch.int32, device=ta.device)
    D.label_max_id(ta, mx[0:1])
    D.label_max_id(tb, mx[1:2])
    max_a, max_b = (int(v) for v in mx.cpu().numpy().view(np.uint32))
    capacity = _initial_capacity(max_a, max_b, a.size)
    limit = _pow2(2 * a.size + 1024)
    while True:
        keys, counts, n_out = D.label_overlap(ta, tb, capacity)
        n_pairs, dropped = (int(v) for v in n_out.cpu().numpy())
        if dropped == 0:
            break
        if capacity >= limit:
            raise D._lib.PlatyMatchError("pm_label_overlap: %d voxels found no table slot at capacity %d" %
                                         (dropped, capacity))
        capacity *= 4
    skeys, order = torch.sort(keys[:n_pairs])
    out = torch.stack([skeys, counts[:n_pairs][order]]).cpu().numpy()
    return out[0] >> 32, out[0] & 0xFFFFFFFF, out[1]


def label_contingency(labels_a, labels_b):
    """Overlap table of two label volumes of one shape, on the GPU (pm_label_overlap).

    labels_a, labels_b  3-D integer volumes (int32 and uint16 are read directly; other integer dtypes go through int32,
                        ids above 2^31 - 1 are refused).  Ids <= 0 count as background (0).
    Returns (ids_a, ids_b, counts), int64 arrays sorted by (a, b): every pair (a, b) != (0, 0) that meets at some voxel
    and its voxel count, i.e. np.unique of the keys a << 32 | b with the (0, 0) entry removed.  The background rows
    (a, 0) and (0, b) are included, so the table's row and column sums are the instance sizes.
    Synchronises with the host 5 times (the upload of each volume, the largest ids, the pair count, the result copy),
    plus once per rerun after a table overflow (at most a few, and only when a volume pair has far more distinct pairs
    than ids).
    """
    a, b = _check_pair(labels_a, labels_b)
    return _contingency(a, b)


def _ratio(n, d):
    return float(n) / float(d) if d else 0.0


def _sizes(ids, counts):
    _, inv = np.unique(ids, return_inverse=True)
    return np.bincount(inv, weights=counts.astype(np.float64)).astype(np.int64)[inv]


def _matching_problem(ids_t, ids_p, iou, threshold):
    """The assignment problem of one threshold from the foreground pairs (ids_t, ids_p, iou): (rows_are_true, row_ids,
    col_ids, r, c, cost, iou) with cost[k] = float32(-(1 + iou[k] / (2K))) at (r[k], c[k]) for each admissible pair k,
    0 elsewhere; rows are the side with fewer ids that have an admissible partner.  None when no pair is admissible."""
    adm = iou >= threshold
    if not adm.any():
        return None
    t, p, v = ids_t[adm], ids_p[adm], iou[adm]
    ut, up = np.unique(t), np.unique(p)
    rows_true = ut.size <= up.size                  # scipy solves the transpose of a tall matrix
    if max(ut.size, up.size) > LAP_MAX_COLUMNS:
        raise ValueError("%d instances with an admissible partner at IoU >= %g: more than the assignment's %d columns"
                         % (max(ut.size, up.size), threshold, LAP_MAX_COLUMNS))
    k = min(ut.size, up.size)
    cost = (-(1.0 + v / (2.0 * k))).astype(np.float32)
    rt, rp = np.searchsorted(ut, t), np.searchsorted(up, p)
    if rows_true:
        return True, ut, up, rt, rp, cost, v
    return False, up, ut, rp, rt, cost, v


def _solve(torch, problem):
    """One assignment on the GPU (D.lap_solve) -> (assigned row indices, their columns, total cost).  Two host
    synchronisations: one upload of the admissible pairs, one copy of the result."""
    _, row_ids, col_ids, r, c, cost, _ = problem
    nr, nc = row_ids.size, col_ids.size
    # (rows, columns, costs) in one float32 upload: indices stay below 24576, exact in float32
    pairs = torch.from_numpy(np.stack([r, c, cost]).astype(np.float32)).cuda()
    idx = pairs[:2].long()
    dense = torch.zeros((nr, (nc + 3) // 4 * 4), dtype=torch.float32, device="cuda")
    dense[idx[0], idx[1]] = pairs[2]
    col4row, total, stats = D.lap_solve(dense, nr, nc)
    res = torch.cat([col4row[0].to(torch.int64), stats[0], total.view(torch.int64)]).cpu().numpy()
    if res[nr + 4] != 0:
        raise D._lib.PlatyMatchError("pm_lap_solve: status %d" % res[nr + 4])
    return np.arange(nr), res[:nr], float(res[-1:].view(np.float64)[0])


def match_labels(labels_true, labels_pred, thresholds=(0.5,)):
    """Compare a predicted label volume with a true one of the same shape, on the GPU.

    One table pass (`label_contingency`), then one exact assignment (the registration's LAP kernel) per threshold.
    Returns a dict:
      dice, jaccard      foreground overlap 2 n_fg / (|A_fg| + |B_fg|) and n_fg / (|A_fg| + |B_fg| - n_fg), where n_fg
                         counts the voxels with a > 0 and b > 0
      n_true, n_pred     non-empty ids of each volume
      per_threshold      one dict per threshold t: threshold, tp, fp = n_pred - tp, fn = n_true - tp, precision,
                         recall, accuracy = tp / (tp + fp + fn), f1, mean_matched_iou, matched = (id_true, id_pred, iou)
                         arrays sorted by id_true, and cost (the assignment's total); a ratio with a zero denominator is 0
    Matching: a pair is admissible when IoU >= t.  Only ids with an admissible partner enter the matrix, the side with
    fewer of them as rows; an admissible pair costs float32(-(1 + IoU / (2K))), K = min(rows, columns), any other 0.
    The optimum therefore has the most admissible pairs first and the largest summed IoU second (exactly, for the
    float32 matrix), and tp counts its admissible pairs.  A threshold at which more than 24576 ids of either volume have
    an admissible partner is refused with a ValueError (the assignment kernel's column limit); ids without one never
    count towards it.
    Synchronises with the host 5 times for the table (plus once per overflow rerun) and twice per threshold that has an
    admissible pair; the volume size does not change that number.
    """
    a, b = _check_pair(labels_true, labels_pred)
    ths = [float(t) for t in np.atleast_1d(np.asarray(thresholds, dtype=np.float64))]
    if not ths or not all(0.0 < t <= 1.0 for t in ths):
        raise ValueError("thresholds must lie in (0, 1], got %r" % (thresholds,))
    ia, ib, n = _contingency(a, b)
    size_a, size_b = _sizes(ia, n), _sizes(ib, n)
    n_true, n_pred = np.unique(ia[ia > 0]).size, np.unique(ib[ib > 0]).size
    fg = (ia > 0) & (ib > 0)
    n_fg = int(n[fg].sum())
    a_fg, b_fg = int(n[ia > 0].sum()), int(n[ib > 0].sum())
    t_ids, p_ids, nn = ia[fg], ib[fg], n[fg]
    iou = nn / (size_a[fg] + size_b[fg] - nn).astype(np.float64)
    out = {"dice": _ratio(2 * n_fg, a_fg + b_fg), "jaccard": _ratio(n_fg, a_fg + b_fg - n_fg),
           "n_true": n_true, "n_pred": n_pred, "per_threshold": []}
    torch = None
    for t in ths:
        problem = _matching_problem(t_ids, p_ids, iou, t)
        mt = mp = np.zeros(0, dtype=np.int64)
        mv = np.zeros(0, dtype=np.float64)
        total = 0.0
        if problem is not None:
            torch = torch or D._torch()
            rows_true, row_ids, col_ids, r, c, _, v = problem
            rows, cols, total = _solve(torch, problem)
            # the assigned pairs that are admissible, found among the admissible pairs by the key row * ncols + col
            adm_key = r * col_ids.size + c
            order = np.argsort(adm_key)
            got = rows * col_ids.size + cols
            pos = np.minimum(np.searchsorted(adm_key[order], got), order.size - 1)
            hit = adm_key[order][pos] == got
            mv = v[order[pos[hit]]]
            mr, mc = row_ids[rows[hit]], col_ids[cols[hit]]
            mt, mp = (mr, mc) if rows_true else (mc, mr)
            srt = np.argsort(mt)
            mt, mp, mv = mt[srt], mp[srt], mv[srt]
        tp = int(mt.size)
        fp, fn = n_pred - tp, n_true - tp
        out["per_threshold"].append({
            "threshold": t, "tp": tp, "fp": fp, "fn": fn, "precision": _ratio(tp, tp + fp), "recall": _ratio(tp, tp + fn),
            "accuracy": _ratio(tp, tp + fp + fn), "f1": _ratio(2 * tp, 2 * tp + fp + fn),
            "mean_matched_iou": _ratio(mv.sum(), tp), "matched": (mt, mp, mv), "cost": total})
    return out


def assign_by_distance(points_a, points_b):
    """linear_sum_assignment(cdist(a.T, b.T)) for 3 x Na / 3 x Nb clouds (:1032-1033, :1038-1039, :1050-1051):
    (row_ind ascending, col_ind) as scipy returns them."""
    torch = D._torch()
    a, b = D.to_device_points(points_a), D.to_device_points(points_b)
    na, nb = a.shape[0], b.shape[0]
    if na <= nb:
        cost = D.cdist(a, b)
        col4row, _, st = D.lap_solve(cost.unsqueeze(0), na, nb)
        rows, cols = np.arange(na, dtype=np.int64), col4row[0].cpu().numpy().astype(np.int64)
    else:                                   # scipy solves the transpose; pairs are reported by ascending row
        cost = D.cdist(b, a)
        col4row, _, st = D.lap_solve(cost.unsqueeze(0), nb, na)
        r = col4row[0].cpu().numpy().astype(np.int64)
        order = np.argsort(r)
        rows, cols = r[order], np.arange(nb, dtype=np.int64)[order]
    if int(st[0, 4].item()) != 0:
        raise ValueError("cost matrix is infeasible")
    return rows, cols


def calculate_metrics(moving_keypoints, moving_keypoint_ids, moving_detections, moving_ids,
                      fixed_keypoints, fixed_keypoint_ids, fixed_detections, fixed_ids,
                      transform_matrix_1, transform_matrix_2=None):
    """reference _dock_widget.py:1030-1080 -> (matching_accuracy, average_registration_error) as floats.

    keypoints / detections are 3 x K and 3 x N (zyx) with their id vectors; the moving cloud is mapped through
    transform_matrix_1 and then transform_matrix_2 (identity if omitted; :1044-1046, combined at :1028).
    """
    from .estimate_transform.apply_transform import apply_affine_transform
    moving_keypoint_ids, fixed_keypoint_ids = np.asarray(moving_keypoint_ids), np.asarray(fixed_keypoint_ids)
    moving_ids, fixed_ids = np.asarray(moving_ids), np.asarray(fixed_ids)
    t1 = np.asarray(transform_matrix_1, dtype=np.float64)
    t2 = np.eye(4) if transform_matrix_2 is None else np.asarray(transform_matrix_2, dtype=np.float64)
    # first associate keypoints with detections (:1032-1042)
    r, c = assign_by_distance(moving_keypoints, moving_detections)
    moving_dictionary = {moving_keypoint_ids[i]: moving_ids[c[k]] for k, i in enumerate(r)}
    r, c = assign_by_distance(fixed_keypoints, fixed_detections)
    fixed_dictionary = {fixed_keypoint_ids[i]: fixed_ids[c[k]] for k, i in enumerate(r)}
    # transformed moving detections against fixed detections (:1044-1051)
    moved = apply_affine_transform(apply_affine_transform(moving_detections, t1), t2)
    row_indices, col_indices = assign_by_distance(moved, fixed_detections)
    row_ids, col_ids = moving_ids[row_indices], fixed_ids[col_indices]
    hits = 0
    for key in moving_dictionary.keys():                                            # :1058-1062
        if key in fixed_dictionary.keys():
            if np.any(col_ids[np.where(row_ids == moving_dictionary[key])] == fixed_dictionary[key]):
                hits += 1
    accuracy = hits / len(fixed_dictionary.keys())                                  # :1067
    combined = np.matmul(t2, t1)                                                    # :1028
    moved_kp = apply_affine_transform(moving_keypoints, combined)
    distance = 0.0
    fk = np.asarray(fixed_keypoints, dtype=np.float64)[:3].transpose()
    for i in range(moved_kp.shape[1]):                                              # :1072-1076
        sel = fk[np.where(fixed_keypoint_ids == moving_keypoint_ids[i])]
        distance += np.linalg.norm(sel - moved_kp.transpose()[i, :])
    return accuracy, distance / len(moving_dictionary.keys())                        # :1079
