"""Particle sharding plan of the multi-GPU path (SURVEY.md section 8e), host-side mirror of the device code
(pft_tracker_kernels.cuh: raw_slot, the item loop of weight_lists_kernel).

Particle i is weighted by rank i % R.  Every rank owns slice_cap = ceil(n_cap / R) slots of the gathered
raw-weight buffer [R][slice_cap]; particle i sits at row i % R, column i // R."""
import numpy as np


def owner(i, nranks):
    return i % nranks


def slice_cap(n_cap, nranks):
    return (n_cap + nranks - 1) // nranks


def local_particles(n, nranks, rank):
    """Global indices of the particles rank `rank` weights, in the order of its slice."""
    return np.arange(rank, n, nranks)


def raw_slot(i, nranks, cap):
    return (i % nranks) * cap + i // nranks


def assemble(gathered, n, nranks):
    """[R][slice_cap] all-gather result -> raw weights in particle order."""
    g = np.asarray(gathered).reshape(nranks, -1)
    i = np.arange(n)
    return g[i % nranks, i // nranks]
