"""fit_cluster and the label-equality mask builders - drop-in for
/root/reference/clustering/cluster_masks.py plus the four mask call sites that consume its labels.

The reference file holds only `fit_cluster` (cluster_masks.py:38-98); the positive / negative masks
are built inline at
    loss/triplet_loss.py:136-142, 254-261, 291-297   per-label positives / negatives in a batch
    models/infoNCE.py:281-283                         UberNCE  B x (1+K) positive mask
    datasets/triplets_dataset.py:99-104               label -> row-indices table
They are exported here as positive_mask / negative_mask / queue_positive_mask / group_by_label /
label_to_indices, each one launch of a kernel in csrc/masks.cu or csrc/cc.cu.
"""
import numpy as np
import torch

from .. import backend as _backend
from .finch import FINCH
from .spherical_kmeans import SphericalKMeans

_METHODS = ['DBSCAN', 'Agglomerative', 'OPTICS', 'kmeans', 'spherical_kmeans', 'finch']


def fit_cluster(embeddings, method='Agglomerative', k=1000, l2normalize=True, finch_partition=0):
    """cluster_masks.py:38-98.  method='finch' (the one the shipped configs use,
    config/custom_configs/resnet_ucf_itercluster_flow.yaml:49-50) and method='spherical_kmeans'
    (SphericalKMeans(n_clusters=k), clustering/spherical_kmeans.py) run on the B200 path; the sklearn methods
    are outside it and raise NotImplementedError.  l2normalize has no effect on spherical_kmeans, which
    normalises the rows itself.

    embeddings: torch tensor [N, D] (CPU as the reference passes it, or already on the GPU - then the
    host round trip of cluster_masks.py:80 is skipped).  Returns int32 labels [N] (numpy)."""
    assert(method in _METHODS)                                       # cluster_masks.py:42-43
    print("Clustering with {}...".format(method))
    if method == 'spherical_kmeans':
        if isinstance(embeddings, torch.Tensor):
            embeddings = embeddings.detach()
        labels = SphericalKMeans(n_clusters=k).fit(embeddings).labels_
        print("Fitted " + str(k) + " clusters with " + str(method))
        return labels
    if method != 'finch':
        raise NotImplementedError("method=%r is not on the B200 hot path; use the reference for it" % method)
    if isinstance(embeddings, torch.Tensor):
        embeddings = embeddings.detach()
    c, num_clust, req_c = FINCH(embeddings, distance='cosine')      # cluster_masks.py:81
    labels = c[:, finch_partition]                                   # cluster_masks.py:83-85
    n_clusters = num_clust[finch_partition]
    print('Taking partition {} from finch'.format(finch_partition))
    print("Fitted " + str(n_clusters) + " clusters with " + str(method))
    return labels


# ---------------------------------------------------------------------------------------------
# masks
# ---------------------------------------------------------------------------------------------
def _labels_on_device(be, labels):
    if isinstance(labels, torch.Tensor):
        return be.to_device(labels.detach(), torch.int64)
    return be.to_device(np.asarray(labels), torch.int64)


def positive_mask(a_labels, b_labels=None, backend=None):
    """mask[i, j] = (a_labels[i] == b_labels[j]) as a torch.bool CUDA tensor [len(a), len(b)].
    With b_labels=None: the in-batch mask labels x labels (triplet_loss.py:136-138, `labels == label`
    for every label at once)."""
    be = backend or _backend.default_backend()
    a = _labels_on_device(be, a_labels)
    b = a if b_labels is None else _labels_on_device(be, b_labels)
    return be.label_mask(a, b)


def negative_mask(a_labels, b_labels=None, backend=None):
    """mask[i, j] = (a_labels[i] != b_labels[j]) - torch.logical_not(label_mask) of
    triplet_loss.py:142, 260, 296, without the intermediate."""
    be = backend or _backend.default_backend()
    a = _labels_on_device(be, a_labels)
    b = a if b_labels is None else _labels_on_device(be, b_labels)
    return be.label_mask(a, b, negate=True)


def queue_positive_mask(k_label, queue_label, backend=None):
    """models/infoNCE.py:281-283: [B, 1+K] bool, column 0 all True (the query's own key), then
    k_label[b] == queue_label[k]."""
    be = backend or _backend.default_backend()
    return be.label_mask(_labels_on_device(be, k_label), _labels_on_device(be, queue_label), prepend_ones=True)


def positive_mask_bits(a_labels, b_labels=None, backend=None):
    """Bit-packed positive mask: int32 [len(a), ceil(len(b)/32)], bit j of word w = column 32 w + j."""
    be = backend or _backend.default_backend()
    a = _labels_on_device(be, a_labels)
    b = a if b_labels is None else _labels_on_device(be, b_labels)
    return be.label_mask_bits(a, b)


def group_by_label(labels, num_labels=None, backend=None):
    """CSR grouping of rows by dense label 0..C-1: (order int32 [N], offsets int32 [C+1]); the rows of
    label c are order[offsets[c]:offsets[c+1]], ascending - what np.where(data_labels == c)[0] yields
    (datasets/triplets_dataset.py:104) at O(N) instead of O(N * C)."""
    be = backend or _backend.default_backend()
    if isinstance(labels, torch.Tensor):
        lab = be.to_device(labels.detach(), torch.int32)
    else:
        lab = be.to_device(np.asarray(labels).astype(np.int32, copy=False), torch.int32)
    if num_labels is None:
        num_labels = int(lab.max().item()) + 1
    return be.group_by_label(lab, int(num_labels))


def label_to_indices(data_labels, backend=None):
    """datasets/triplets_dataset.py:99-104 for arbitrary (not necessarily dense) integer labels:
    {label: ascending row indices}.  Dense relabelling (slic_dense_labels) and grouping both run on the device."""
    be = backend or _backend.default_backend()
    if isinstance(data_labels, torch.Tensor):
        lab = be.to_device(data_labels.detach().reshape(-1), torch.int32)
    else:
        lab = be.to_device(np.asarray(data_labels).reshape(-1).astype(np.int32, copy=False), torch.int32)
    dense, uniq, count = be.dense_labels(lab)                        # np.unique(..., return_inverse=True) on the device
    order, offsets = be.group_by_label(dense, count)
    order, offsets, uniq = be.to_host(order), be.to_host(offsets), be.to_host(uniq)
    return {uniq[c].item(): order[offsets[c]:offsets[c + 1]].astype(np.int64) for c in range(count)}
