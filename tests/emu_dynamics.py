"""The per-env dynamics table's fields (include/prb.h prb_dynamics), as EmuSim(table=...) holds them for the emulated
setup kernel (its `dyn` argument in csrc/prb_stream.cuh) and the randomization kernel (csrc/prb_dynamics.cuh).  CPU
tests only."""
import numpy as np

# the table's fields in include/prb.h prb_dynamics order, with the model field each one overrides
FIELDS = ['lateral_friction', 'spinning_friction', 'mass', 'local_inertia_diagonal', 'linear_damping', 'angular_damping']
MODEL_FIELD = {'lateral_friction': 'col_friction', 'spinning_friction': 'col_spin', 'mass': 'free_mass',
               'local_inertia_diagonal': 'free_inertia', 'linear_damping': 'free_lin_damp', 'angular_damping': 'free_ang_damp'}
RANGE_FIELDS = ['lateral_friction', 'spinning_friction', 'mass', 'linear_damping', 'angular_damping']


def model_table(m, N):
    """Every env's row holding the model's values, the (float) casts of csrc/prb_convert.h."""
    nc, nf = int(m['n_col']), int(m['n_free'])
    f = lambda k, n: np.asarray(m[MODEL_FIELD[k]], np.float64)[:n].astype(np.float32)
    return {'lateral_friction': np.tile(f('lateral_friction', nc), (N, 1)),
            'spinning_friction': np.tile(f('spinning_friction', nc), (N, 1)),
            'mass': np.tile(f('mass', nf), (N, 1)),
            'local_inertia_diagonal': np.tile(f('local_inertia_diagonal', 3 * nf).reshape(nf, 3), (N, 1, 1)),
            'linear_damping': np.tile(f('linear_damping', nf), (N, 1)),
            'angular_damping': np.tile(f('angular_damping', nf), (N, 1))}
