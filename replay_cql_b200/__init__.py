"""replay_cql_b200 -- B200-native CQL recommender hot path behind RePlay's plug-in API.

Only what the path needs lives here:

* ``csrc/``        hand-written sm_100a CUDA kernels + the C-ABI library (``include/cql_b200.h``)
* ``_lib``         ctypes binding of that library (fails loudly without it / without a GPU)
* ``layout``       flat parameter layout shared with the kernels
* ``engine``       host driver: device state, update loop, data-parallel step, scoring
* ``mdp``          MDP builder (log -> episode-ordered transitions)
* ``recommender``  pandas/pyarrow mirror of RePlay's ``Recommender`` template methods
* ``models``       ``CQL`` -- the drop-in model class
* ``model_handler`` ``save`` / ``load`` with the reference's directory layout
* ``ope``          ``FQE`` -- fitted Q evaluation of a trained ``CQL`` policy (``replay_cql_b200.FQE``)
"""
__version__ = "0.1.0"


def __getattr__(name):
    # imported on first use: the package itself stays light to import
    if name == "FQE":
        from .ope import FQE
        return FQE
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
