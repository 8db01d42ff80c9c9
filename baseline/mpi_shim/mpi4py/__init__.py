"""Minimal mpi4py-compatible shim (NOT product code).

mpi4py / mpirun cannot be installed offline in this environment (SURVEY.md fact 10), so
the UNMODIFIED reference (installed under oracle/_ref) is driven through this shim: it
implements exactly the mpi4py surface the reference touches (SURVEY.md section 2.4, C1-C11) on
top of torch.distributed's gloo backend (host memory, like MPI).  World size 1 needs no
process group at all."""
from . import MPI  # noqa: F401
