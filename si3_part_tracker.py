#!/usr/bin/env python3
"""SITRACK ice particle tracker -- B200 drop-in for the reference's `si3_part_tracker.py`.

Same command line (-i -m -s required; -k -e -F -N -p), same file-name conventions, same
seeding cache (`./seed/Initialized_buoys_<Seed>_<CONF>.npz`) and the same two output files
(`./nc/..._tracking_...` with -F, and the 2-record `..._tracking12_...`), but the seeding
loop (reference tracking.py:120-160) and the records x buoys loop
(reference si3_part_tracker.py:361-496) run on the GPU through sitrack_b200.TrackEngine.
Inputs may be netCDF (needs netCDF4) or the `.npz` equivalents described in
sitrack_b200/ncio.py.  Plotting (-p) is accepted and ignored: the plotting stack (mojito,
cartopy) is outside the scope of this path.

Several GPUs: `torchrun --nproc-per-node N si3_part_tracker.py ...` (one process per GPU).  Rank 0 does the
seeding stage; every rank then tracks its contiguous block of buoys (they never interact, reference :378-488)
with its own replica of the grid and of each record, and rank 0 collects the rows and writes the files.
"""
import os
from os import path, makedirs
from re import split
from sys import exit

import numpy as np

import sitrack_b200 as sit
from sitrack_b200 import epoch2clock as e2c

idebug = 0
rdt = 3600.          # time step [s] of the model output used (reference :31)
iUVstrategy = 1      # 0: mean of the two faces, 1: nearest U / nearest V point (reference :37)


def __argument_parsing__():
    import argparse as ap
    parser = ap.ArgumentParser(description='SITRACK ICE PARTICULES TRACKER')
    rq = parser.add_argument_group('required arguments')
    rq.add_argument('-i', '--fsi3', required=True, help='output file of SI3 containing ice velocities ans co')
    rq.add_argument('-m', '--fmmm', required=True, help='model `mesh_mask` file of NEMO config used in SI3 run')
    rq.add_argument('-s', '--fsdg', required=True, help='seeding file')
    parser.add_argument('-k', '--krec', type=int, default=0, help='record of seeding file to use to seed from')
    parser.add_argument('-e', '--dend', default=None, help='date at which to stop')
    parser.add_argument('-F', '--fxdt', action="store_true", help='fixed tracking time (1D time array)')
    parser.add_argument('-N', '--ncnf', default='NANUK4', help='name of the horizontak NEMO config used')
    parser.add_argument('-p', '--plot', type=int, default=0, help='(ignored) how often we plot the positions on a map')
    parser.add_argument('--device', type=int, default=None, help='CUDA device (default: LOCAL_RANK or 0)')
    parser.add_argument('--uvstrategy', type=int, default=iUVstrategy, choices=[0, 1])
    parser.add_argument('--scheme', default='euler', choices=['euler', 'rk2', 'rk4'],
                        help='time stepping: euler = upstream behaviour (default); rk2/rk4 = optional physics (st_step_ext)')
    parser.add_argument('--interp', default='pick', choices=['pick', 'linear'],
                        help='velocity at the buoy: pick = upstream face pick (default); linear = C-grid linear (st_step_ext)')
    parser.add_argument('--hops', type=int, default=1, help='cell boundaries a buoy may cross per record (upstream: 1)')
    parser.add_argument('--sort', action="store_true",
                        help='store and write the buoys in cell-major order (much faster gathers on large clouds); the '
                             'output files then list the buoys, with their IDs, in that order instead of seed order')
    parser.add_argument('--no-chunk', action="store_true",
                        help='small clouds: one kernel launch per record (streaming) instead of one per chunk of records')
    parser.add_argument('--rows', default='f4', choices=['f4', 'f8'],
                        help='dtype of the trajectory rows copied off the GPU: f4 = the dtype the output files store (default), f8 = full in-memory arrays as upstream')
    parser.add_argument('--deform', type=float, default=None, metavar='HOURS',
                        help='also compute sea-ice deformation (divergence, shear, vorticity) of buoy triangles over '
                             'windows of HOURS (a multiple of the model time step) on the GPU, into ./nc/..._deformation_...')
    parser.add_argument('--deform-maxedge', type=float, default=None, metavar='KM',
                        help='with --deform: drop triangles with an edge longer than KM (default: twice the median edge)')
    parser.add_argument('--deform-scales', type=float, nargs=2, default=None, metavar=('L0_KM', 'LEVELS'),
                        help='with --deform: also coarse-grain the triangles over LEVELS levels of material boxes of side '
                             'L0_KM * 2^s and write per-scale statistics (n, means of L_eff and eps_tot^q, histograms) '
                             'of every window into ./nc/..._deformation-scaling_...')
    parser.add_argument('--deform-grid', type=float, nargs=2, default=None, metavar=('L0_KM', 'LEVELS'),
                        help='with --deform: also coarse-grain the triangles over the fixed cells of a grid of side L0_KM * 2^s '
                             '(LEVELS levels) covering the model\'s T-points, binned every window by mid-time centroid, and '
                             'write per-level fields into ./nc/..._deformation-grid_... and per-scale statistics into '
                             './nc/..._deformation-grid-scaling_...')
    parser.add_argument('--dispersion', type=float, nargs=2, default=None, metavar=('HOURS', 'LAGS'),
                        help='also compute two-particle dispersion of buoy pairs on the GPU: origins every HOURS (a multiple '
                             'of the model time step), lags of 1..LAGS windows, per-lag and per-separation-class statistics '
                             'of every window into ./nc/..._dispersion_...')
    parser.add_argument('--dispersion-pairs', type=float, nargs=3, default=None, metavar=('N', 'R_MIN_KM', 'R_MAX_KM'),
                        help='with --dispersion: N random draws of pairs at log-uniform separations in [R_MIN_KM, R_MAX_KM] '
                             '(default: one draw per buoy, 10 to 1000 km)')
    parser.add_argument('--fsle', type=float, default=None, metavar='HOURS',
                        help='also compute finite-size Lyapunov exponents of buoy pairs on the GPU: the pairs are sampled '
                             'every HOURS (a multiple of the model time step) and the exit times between separation '
                             'thresholds of every window go into ./nc/..._fsle_...')
    parser.add_argument('--fsle-deltas', type=float, nargs=3, default=None, metavar=('D0_KM', 'ALPHA', 'K'),
                        help='with --fsle: K (2..64) thresholds D0_KM * ALPHA^j (default: 2 km, sqrt(2), 19)')
    parser.add_argument('--fsle-pairs', type=float, nargs=3, default=None, metavar=('N', 'R_MIN_KM', 'R_MAX_KM'),
                        help='with --fsle: N random draws of pairs at log-uniform separations in [R_MIN_KM, R_MAX_KM] '
                             '(default: one draw per buoy, 10 to 1000 km)')
    parser.add_argument('--sample', nargs='+', default=None, metavar='VAR',
                        help='also sample these SI3 T-cell variables (e.g. siconc sithic) along the trajectories on the GPU '
                             'and write them, per sampled row and buoy, into ./nc/..._sampled_...')
    parser.add_argument('--sample-every', type=float, default=None, metavar='HOURS',
                        help='with --sample: sample every HOURS (a multiple of the model time step; default: every record)')
    parser.add_argument('--sample-interp', default=None, choices=['cell', 'bilinear'],
                        help='with --sample: the host cell\'s value (cell, default) or the bilinear interpolation '
                             'between the four T-points around the buoy (bilinear)')
    parser.add_argument('--connect', type=float, default=None, metavar='HOURS',
                        help='also count buoy transits between the regions of a label map on the GPU: the buoys\' host '
                             'cells are sampled every HOURS (a multiple of the model time step) and per-window starts, '
                             'ends, transitions, source-to-region counts and first-arrival times go into '
                             './nc/..._connectivity_...')
    parser.add_argument('--connect-regions', nargs=2, default=None, metavar=('FILE', 'VAR'),
                        help='with --connect: the (y,x) variable VAR of FILE (netCDF or .npz) labels the T-cells with '
                             'regions 1..31 (0 or a masked value: in no region)')
    args = parser.parse_args()
    print('')
    print(' *** SI3 file to get ice velocities from => ', args.fsi3)
    print(' *** SI3 `mesh_mask` metrics file        => ', args.fmmm)
    print(' *** Seeding file and record to use      => ', args.fsdg, args.krec)
    if args.dend:
        print(' *** Overidding date at which to stop =>', args.dend)
    if args.ncnf:
        print(' *** Name of the horizontak NEMO config used => ', args.ncnf)
    return args


def seed_name_info(fNCseedBN):
    """`csfkm`, `cdtbin` from the seeding file name (reference :115-148)."""
    csfkm = ''
    stem = split(r'\.', fNCseedBN)[0]
    parts = split('_', stem)
    if parts[2] in ['nemoTsi3', 'nemoTmm', 'sidfex']:
        print('\n *** Seems to be an idealized seeding of type "' + parts[2] + '"')
        cdtbin = '_idlSeed'
        for ii in [1, 2, 3]:
            ckm = '_' + parts[-ii]
            if ckm[-2:] == 'km':
                csfkm = ckm
                break
    else:
        lok, itst = False, 1
        base = split('_', split(r'\.', fNCseedBN)[-2])
        while not lok:
            itst -= 1
            csfkm = '_' + base[itst]
            cdtbin = '_' + base[-3 + itst]
            lok = (csfkm[-2:] == 'km' and cdtbin[1:3] == 'dt') or (cdtbin[1:3] == 'dt' and itst == 0)
            if itst < -4:
                print('ERROR: we could not figure out `csfkm` and `cdtbin` from file name!', csfkm, cdtbin)
                exit(0)
        if itst == 0:
            csfkm = ''
    return csfkm, cdtbin


def record_windows(zTpos, nP, kstrt, kstop, ztime_model, iTmA, iTmB):
    """First/last model record per buoy without -F (reference :264-312)."""
    z1st = np.zeros(nP, dtype=int) + kstrt
    zLst = np.zeros(nP, dtype=int) + kstop
    (n2, nB) = np.shape(zTpos)
    if n2 != 2 or nP != nB:
        print('ERROR: wrong shape for the 2D time array `zTpos`! `n2,nB`, vs `nP`:', n2, nB, nP)
        exit(0)
    half = int(rdt / 2)
    for jb in np.where(zTpos[0, :] >= iTmA + half)[0]:
        (idx,) = np.where(ztime_model + half < zTpos[0, jb])
        z1st[jb] = idx[-1] + 1
    for jb in np.where(zTpos[1, :] < iTmB - half)[0]:
        (idx,) = np.where(ztime_model - half > zTpos[1, jb])
        zLst[jb] = idx[0] - 1
    return z1st, zLst


def window_records(flag, hours):
    """HOURS of `flag` -> records per window; ERROR and exit when it is not a positive multiple of the model time
    step."""
    n = hours * 3600. / rdt
    if not (hours > 0 and abs(n - round(n)) < 1e-9 and round(n) >= 1):
        print('ERROR: %s HOURS must be a positive multiple of the model time step (%g h), got %g' % (flag, rdt / 3600., hours))
        exit(0)
    return int(round(n))


def deform_records(hours, world):
    """--deform HOURS -> records per deformation window (None without the flag); ERROR and exit when it is not a
    positive multiple of the model time step, or under torchrun (triangles would cross the ranks' shards)."""
    if hours is None:
        return None
    if world > 1:
        print('ERROR: --deform is not available with several processes (WORLD_SIZE > 1): triangles would cross ranks')
        exit(0)
    return window_records('--deform', hours)


def deform_levels_args(flag, levels, hours):
    """`flag` L0_KM LEVELS (--deform-scales, --deform-grid) -> (L0_km, levels) or None; ERROR and exit without
    --deform, with L0 <= 0, or with LEVELS not an integer in 1..20."""
    if levels is None:
        return None
    L0, lev = levels
    if hours is None:
        print('ERROR: %s needs --deform HOURS' % flag)
        exit(0)
    if not L0 > 0:
        print('ERROR: %s L0_KM must be positive, got %g' % (flag, L0))
        exit(0)
    if lev != int(lev) or not 1 <= lev <= sit.MAX_LEVELS:
        print('ERROR: %s LEVELS must be an integer in 1..%d, got %g' % (flag, sit.MAX_LEVELS, lev))
        exit(0)
    return L0, int(lev)


def dispersion_args(disp, pairs, world):
    """--dispersion HOURS LAGS [--dispersion-pairs N R_MIN_KM R_MAX_KM] -> (records per window, lags, N or None,
    r_min, r_max) or None; ERROR and exit when HOURS is not a positive multiple of the model time step, LAGS is not an
    integer in 1..MAX_LAGS, N < 1, R_MIN <= 0 or R_MAX <= R_MIN, --dispersion-pairs comes without --dispersion, or under
    torchrun (pairs would cross the ranks' shards)."""
    if disp is None:
        if pairs is not None:
            print('ERROR: --dispersion-pairs needs --dispersion HOURS LAGS')
            exit(0)
        return None
    hours, lags = disp
    if world > 1:
        print('ERROR: --dispersion is not available with several processes (WORLD_SIZE > 1): pairs would cross ranks')
        exit(0)
    n = window_records('--dispersion', hours)
    if lags != int(lags) or not 1 <= lags <= sit.MAX_LAGS:
        print('ERROR: --dispersion LAGS must be an integer in 1..%d, got %g' % (sit.MAX_LAGS, lags))
        exit(0)
    N, r_min, r_max = (None, 10.0, 1000.0) if pairs is None else pairs
    if N is not None and (N != int(N) or N < 1):
        print('ERROR: --dispersion-pairs N must be a positive integer, got %g' % N)
        exit(0)
    if not (r_min > 0 and r_max > r_min and np.isfinite(r_max)):
        print('ERROR: --dispersion-pairs needs 0 < R_MIN_KM < R_MAX_KM, got %g %g' % (r_min, r_max))
        exit(0)
    return n, int(lags), None if N is None else int(N), r_min, r_max


def fsle_args(hours, deltas, pairs, world):
    """--fsle HOURS [--fsle-deltas D0_KM ALPHA K] [--fsle-pairs N R_MIN_KM R_MAX_KM] -> (records per sample, the
    thresholds, N or None, r_min, r_max) or None; ERROR and exit when HOURS is not a positive multiple of the model
    time step, K is not an integer in 2..64, D0 <= 0, ALPHA <= 1 or the thresholds are not finite and increasing,
    N < 1, R_MIN <= 0 or R_MAX <= R_MIN, an option comes without --fsle, or under torchrun (pairs would cross the
    ranks' shards)."""
    if hours is None:
        for flag, v in (('--fsle-deltas', deltas), ('--fsle-pairs', pairs)):
            if v is not None:
                print('ERROR: %s needs --fsle HOURS' % flag)
                exit(0)
        return None
    if world > 1:
        print('ERROR: --fsle is not available with several processes (WORLD_SIZE > 1): pairs would cross ranks')
        exit(0)
    n = window_records('--fsle', hours)
    D0, alpha, K = (2.0, np.sqrt(2.0), 19) if deltas is None else deltas
    if K != int(K) or not 2 <= K <= sit.MAX_THRESHOLDS:
        print('ERROR: --fsle-deltas K must be an integer in 2..%d, got %g' % (sit.MAX_THRESHOLDS, K))
        exit(0)
    if not (D0 > 0 and alpha > 1):
        print('ERROR: --fsle-deltas needs D0_KM > 0 and ALPHA > 1, got %g %g' % (D0, alpha))
        exit(0)
    with np.errstate(over='ignore'):
        d = np.float64(D0) * np.float64(alpha) ** np.arange(int(K), dtype=np.float64)
    if not (np.isfinite(d).all() and (np.diff(d) > 0).all()):
        print('ERROR: --fsle-deltas: the thresholds D0_KM * ALPHA^j are not finite and increasing (last %g)' % d[-1])
        exit(0)
    N, r_min, r_max = (None, 10.0, 1000.0) if pairs is None else pairs
    if N is not None and (N != int(N) or N < 1):
        print('ERROR: --fsle-pairs N must be a positive integer, got %g' % N)
        exit(0)
    if not (r_min > 0 and r_max > r_min and np.isfinite(r_max)):
        print('ERROR: --fsle-pairs needs 0 < R_MIN_KM < R_MAX_KM, got %g %g' % (r_min, r_max))
        exit(0)
    return n, d, None if N is None else int(N), r_min, r_max


def sample_args(names, hours, interp):
    """--sample VAR [VAR ...] [--sample-every HOURS] [--sample-interp cell|bilinear] -> (names, records between sampled
    rows, interp) or None; ERROR and exit when HOURS is not a positive multiple of the model time step, a variable is
    named twice or more than MAX_SAMPLE_FIELDS are named, or an option comes without --sample."""
    if names is None:
        for flag, v in (('--sample-every', hours), ('--sample-interp', interp)):
            if v is not None:
                print('ERROR: %s needs --sample VAR [VAR ...]' % flag)
                exit(0)
        return None
    if len(set(names)) != len(names) or len(names) > sit.MAX_SAMPLE_FIELDS:
        print('ERROR: --sample needs 1..%d distinct variables, got %s' % (sit.MAX_SAMPLE_FIELDS, ' '.join(names)))
        exit(0)
    n = 1 if hours is None else window_records('--sample-every', hours)
    return list(names), n, interp or 'cell'


def check_sample_vars(ds, names):
    """ERROR and exit when a --sample variable is missing from the SI3 file or is not a (t,y,x) variable of the shape
    of u_ice; -> {name: units} of those that have units."""
    ref = tuple(ds.variables['u_ice'].shape)
    units = {}
    for n in names:
        if n not in ds.variables:
            print('ERROR: --sample: variable %s is not in the SI3 file' % n)
            exit(0)
        v = ds.variables[n]
        if tuple(v.shape) != ref:
            print('ERROR: --sample: %s has shape %s, not the (t,y,x) shape %s of u_ice' % (n, tuple(v.shape), ref))
            exit(0)
        u = getattr(v, 'units', None)
        if u is not None:
            units[n] = str(u)
    return units


def connect_args(hours, regions):
    """--connect HOURS --connect-regions FILE VAR -> (records per sample, FILE, VAR) or None; ERROR and exit when one
    comes without the other or HOURS is not a positive multiple of the model time step."""
    if (hours is None) != (regions is None):
        print('ERROR: --connect HOURS and --connect-regions FILE VAR go together')
        exit(0)
    if hours is None:
        return None
    return window_records('--connect', hours), regions[0], regions[1]


def connect_labels(fn, var, shape):
    """The region map VAR of FILE as (u8 labels, R); ERROR and exit when the file or the variable is missing, the
    variable is not `shape` (the model's (y,x)) after taking its first (y,x) plane, or its labels are refused."""
    from sitrack_b200.ncio import _plane
    if not path.exists(fn):
        print('ERROR: --connect-regions: file %s not found' % fn)
        exit(0)
    with sit.open_dataset(fn) as ds:
        if var not in ds.variables:
            print('ERROR: --connect-regions: variable %s is not in %s' % (var, fn))
            exit(0)
        v = ds.variables[var]
        a = _plane(v) if len(v.shape) >= 2 else None
    if a is None or a.shape != tuple(shape):
        print('ERROR: --connect-regions: %s has shape %s, not the (y,x) shape %s of the model grid'
              % (var, tuple(v.shape), tuple(shape)))
        exit(0)
    try:
        return sit.connect.check_labels(a, *shape)
    except ValueError as e:
        print('ERROR: --connect-regions: %s' % e)
        exit(0)


def deform_grid_over(Yt, Xt, L0, levels):
    """The EulerianGrid of side L0 covering the T-points (Yt, Xt) km: origin floor(min / L0) L0 and
    floor((max - origin) / L0) + 1 cells per axis; ERROR and exit when that is more than 2^20 cells a side."""
    origin = np.array([np.floor(np.min(Yt) / L0) * L0, np.floor(np.min(Xt) / L0) * L0])
    shape = [int(np.floor((np.max(A) - o) / L0)) + 1 for A, o in ((Yt, origin[0]), (Xt, origin[1]))]
    if max(shape) > sit.MAX_GRID_SIDE:
        print('ERROR: --deform-grid L0_KM = %g gives %d x %d cells over the model grid, more than %d a side'
              % (L0, shape[0], shape[1], sit.MAX_GRID_SIDE))
        exit(0)
    return sit.EulerianGrid(origin, L0, shape, levels)


def main():
    print('\n##########################################################')
    print('#            SITRACK ICE PARTICULES TRACKER              #')
    print('#                 (sitrack_b200 engine)                  #')
    print('##########################################################\n')
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    args = __argument_parsing__()
    ndeform = deform_records(args.deform, world)
    dscales = deform_levels_args('--deform-scales', args.deform_scales, args.deform)
    dgrid = deform_levels_args('--deform-grid', args.deform_grid, args.deform)
    dspa = dispersion_args(args.dispersion, args.dispersion_pairs, world)
    fsla = fsle_args(args.fsle, args.fsle_deltas, args.fsle_pairs, world)
    smpa = sample_args(args.sample, args.sample_every, args.sample_interp)
    cona = connect_args(args.connect, args.connect_regions)
    dist = None
    if world > 1:
        import torch.distributed as dist                      # host-side plumbing only: gloo over CPU arrays
        dist.init_process_group("gloo")
    cf_uv, cf_mm, fNCseed, jrecSeed, cdate_stop, CONF = args.fsi3, args.fmmm, args.fsdg, args.krec, args.dend, args.ncnf
    lUse2DTime = not args.fxdt
    if args.device is not None:
        sit.config.device = args.device
    if args.plot:
        print(' *** NOTE: -p/--plot is accepted but plotting is not part of sitrack_b200; ignoring.')
    fNCseedBN = path.basename(fNCseed)
    csfkm, cdtbin = seed_name_info(fNCseedBN)
    creskm = csfkm[1:] if csfkm != '' else ''

    idateSeedA, idateSeedB, SeedName, SeedBatch, zTpos = sit.SeedFileTimeInfo(fNCseed, ltime2d=lUse2DTime, iverbose=idebug)
    Nt0, ztime_model, idateModA, idateModB, ModConf, ModExp = sit.ModelFileTimeInfo(cf_uv, iverbose=idebug)

    date_stop = None
    if cdate_stop:
        date_stop = sit.clock2epoch(cdate_stop) if len(cdate_stop) == 19 else sit.clock2epoch(cdate_stop, precision='D', cfrmt='guess')
    elif idateSeedB - idateSeedA >= 3600.:
        date_stop = idateSeedB
    Nt, kstrt, kstop, iTmA, iTmB = sit.GetTimeSpan(rdt, ztime_model, idateSeedA, idateModA, idateModB, iStop=date_stop)
    if Nt < 1:
        print(' QUITTING since no matching model records!')
        exit(0)
    if dspa and Nt // dspa[0] < 1:
        print('ERROR: --dispersion window (%d records) is longer than the run (%d records)!' % (dspa[0], Nt))
        exit(0)
    if fsla and not 1 <= Nt // fsla[0] <= sit.MAX_SAMPLES:
        print('ERROR: --fsle gives %d windows of %d records over the run (%d records): need 1..%d'
              % (Nt // fsla[0], fsla[0], Nt, sit.MAX_SAMPLES))
        exit(0)
    if cona and not 1 <= Nt // cona[0] <= sit.MAX_SAMPLES:
        print('ERROR: --connect gives %d windows of %d records over the run (%d records): need 1..%d'
              % (Nt // cona[0], cona[0], Nt, sit.MAX_SAMPLES))
        exit(0)
    labels = None
    if cona:
        with sit.open_dataset(cf_uv) as ds0:
            labels, nreg = connect_labels(cona[1], cona[2], ds0.variables['u_ice'].shape[-2:])
    sunits = {}
    if smpa:
        with sit.open_dataset(cf_uv) as ds0:
            sunits = check_sample_vars(ds0, smpa[0])
    for cd in ['seed', 'nc', 'npz']:
        makedirs(cd, exist_ok=True)

    imaskt, xlatT, xlonT, xYt, xXt, xYf, xXf, xResKM = sit.GetModelGrid(cf_mm)
    xYv, xXv, xYu, xXu = sit.GetModelUVGrid(cf_mm) if args.uvstrategy == 1 else (None, None, None, None)
    (Nj, Ni) = np.shape(imaskt)
    G = deform_grid_over(xYt, xXt, *dgrid) if dgrid else None

    ds = sit.open_dataset(cf_uv)
    vU, vV, vIC = ds.variables['u_ice'], ds.variables['v_ice'], ds.variables['siconc']

    # ---- initialization / seeding (reference :205-255) ----------------------------------------
    cf_npz_itm = './seed/Initialized_buoys_' + SeedName + '_' + CONF + '.npz'
    if world > 1 and rank != 0:
        dist.barrier()                                            # rank 0 is locating the seeds / writing the cache
    if path.exists(cf_npz_itm):
        print('\n *** We found file ' + cf_npz_itm + ' here! So using it and skipping first stage!')
        with np.load(cf_npz_itm) as data:
            nP = int(data['nP']); xPosG0 = data['xPosG0']; xPosC0 = data['xPosC0']; IDs = data['IDs']
            vJIt = data['vJIt']; VRTCS = data['VRTCS']; idxK = data['idxKeep']
    else:
        print('\n *** We did not find file ' + cf_npz_itm + ' ! => locating the seeds on the GPU...')
        xIC0 = np.asarray(vIC[kstrt, :, :], dtype=np.float32)
        zt, zIDs, XseedG, XseedC = sit.LoadNCdata(fNCseed, krec=jrecSeed, iverbose=idebug)
        print('     => data used for seeding is read at date =', e2c(zt), '\n        (shape of XseedG =', np.shape(XseedG), ')')
        (nP, _) = np.shape(XseedG)
        IDs = np.array(zIDs, dtype=int)
        nPn, xPosG0, xPosC0, IDs, vJIt, VRTCS, idxK = sit.SeedInit(IDs, XseedG, XseedC, xlatT, xlonT, xYf, xXf,
                                                                   xResKM, imaskt, xIceConc=xIC0, iverbose=idebug)
        if nPn < nP:
            print('\n *** `SeedInit()` had to cancel ' + str(nP - nPn) + ' buoys! => updating nP from ' + str(nP) + ' to ' + str(nPn) + '!')
            nP = nPn
        print('\n *** Saving intermediate data into ' + cf_npz_itm + '!')
        np.savez_compressed(cf_npz_itm, nP=nP, xPosG0=xPosG0, xPosC0=xPosC0, IDs=IDs, vJIt=vJIt, VRTCS=VRTCS, idxKeep=idxK)

    if world > 1 and rank == 0:
        dist.barrier()                                            # the cache is on disk: the other ranks may read it

    z1st = zLst = None
    if lUse2DTime:
        z1st, zLst = record_windows(zTpos, nP, kstrt, kstop, ztime_model, iTmA, iTmB)
    if args.sort and nP > 1:
        # cell-major order for everything downstream: state, rows and the files (IDs carried along)
        perm = np.argsort(vJIt[:, 0].astype(np.int64) * Ni + vJIt[:, 1], kind='stable')
        xPosG0, xPosC0, IDs, vJIt = xPosG0[perm], xPosC0[perm], IDs[perm], vJIt[perm]
        if z1st is not None:
            z1st, zLst = z1st[perm], zLst[perm]
        print(' *** --sort: buoys re-ordered by host cell (cell-major); the output files follow that order')
    lo, hi = 0, nP
    if world > 1:
        from sitrack_b200.dist import my_shard
        lo, hi = my_shard(nP, rank, world)
        print(' *** rank %d of %d tracks buoys [%d, %d) of %d' % (rank, world, lo, hi, nP))
    sh = slice(lo, hi)
    cut = lambda a: None if a is None else a[sh]

    # ---- the record loop on the GPU (reference :361-496) -----------------------------------------
    vTime = np.zeros(Nt + 1, dtype=int)
    for jt in range(Nt):
        vTime[jt] = int(ztime_model[jt + kstrt]) - int(rdt / 2.)
    vTime[Nt] = vTime[Nt - 1] + int(rdt)

    def record(k):
        jrec = k + kstrt
        print('\n *** Reading record #' + str(jrec + 1) + '/' + str(Nt0) + ' in SI3 file ==> date =', e2c(vTime[k]),
              '(model:' + e2c(int(ztime_model[jrec])) + ')')
        return vU[jrec, :, :], vV[jrec, :, :], vIC[jrec, :, :]

    def hstr(it):
        c = split(':', e2c(it))[0]
        return c.replace('-', '').replace('_', 'h')
    corgn = 'NEMO-SI3_' + ModConf + '_' + ModExp
    ext = '.npz' if str(cf_uv).endswith('.npz') else '.nc'

    def nc_name(kind, t0, t1):
        return './nc/' + corgn + '_' + kind + '_' + SeedBatch + cdtbin + '_' + hstr(t0) + '_' + hstr(t1) + csfkm + ext

    writers = []                                                  # the per-window files, closed after track()

    def window_sink(n, *wrs):
        """sink(w, a, b, ...) of windows of n records: a into wrs[0], b into wrs[1], ... with the window's dates"""
        writers.extend(wrs)
        return lambda w, *a: [wr.write(w, vTime[w * n], vTime[(w + 1) * n], x) for wr, x in zip(wrs, a)]

    # Trajectory rows are written as they leave the GPU: the reference holds (Nt+1, nP, 2) arrays for the whole run
    # (:326-328), here only the two rows the `tracking12` file needs stay in memory.
    writer = None
    if rank == 0 and not lUse2DTime:
        writer = sit.CloudBuoyWriter(nc_name('tracking', vTime[0], vTime[Nt]), Nt + 1, IDs, with_mask=True, corigin=corgn)
        writer.write(0, vTime[0], xPosC0[:, 0], xPosC0[:, 1], xPosG0[:, 0], xPosG0[:, 1], mask=np.ones(nP, 'i1'))
    z2XY, z2GC, zMSK = np.zeros((2, nP, 2)), np.zeros((2, nP, 2)), np.zeros((2, nP), dtype='i1')
    z2XY[0], z2GC[0], zMSK[0] = xPosC0, xPosG0, 1                # each buoy's first row is its seed (:335-340)
    kN = (zLst - kstrt + 1) if lUse2DTime else np.zeros(nP, dtype=int) + Nt      # row that closes each buoy's window

    def keep_row(k, yx, ll, m):
        """rank 0, whole rows in file order: append to the full-series file, remember the closing rows"""
        if writer is not None:
            writer.write(k + 1, vTime[k + 1], yx[:, 0], yx[:, 1], ll[:, 0], ll[:, 1], mask=m)
        if not lUse2DTime:                                        # reference :376, live: the buoys this record advanced
            print('   *   record ' + str(k + kstrt) + ': number of buoys alive = ' + str(int(np.count_nonzero(m))))
        sel = np.flatnonzero(kN == k + 1)
        z2XY[1, sel], z2GC[1, sel], zMSK[1, sel] = yx[sel], ll[sel], m[sel]

    sample_stash = []                                             # torchrun: samples that go with the next row

    def sink(k, yx, ll, m):
        if world == 1:
            keep_row(k, yx, ll, m)
        else:                                                     # one small gather per record, rank 0 writes
            parts = [None] * world if rank == 0 else None
            dist.gather_object((yx.copy(), ll.copy(), m.copy(), sample_stash[:]), parts, dst=0)
            sample_stash.clear()
            if rank == 0:
                keep_row(k, *[np.concatenate([p[i] for p in parts]) for i in range(3)])
                for i, (js, vals) in enumerate(parts[0][3]):      # every rank samples the same rows
                    smwriter.write(js, vTime[js * smpa[1]],
                                  {n: np.concatenate([p[3][i][1][n] for p in parts]) for n in vals})

    eng = sit.TrackEngine(xYf, xXf, xYu, xXu, xYv, xXv, tmask=imaskt, uv_strategy=args.uvstrategy, rdt=rdt,
                          rmin_conc=sit.rmin_conc, device=sit.config.device)
    eng.set_buoys(xPosC0[sh], vJIt[sh], cut(z1st), cut(zLst))
    # rows come back in the file's dtype (every trajectory variable is f4, ncio.py:153-159)
    physics = None
    if args.scheme != 'euler' or args.interp != 'pick' or args.hops != 1:
        physics = dict(scheme={'euler': 1, 'rk2': 2, 'rk4': 4}[args.scheme], interp=int(args.interp == 'linear'), max_hops=args.hops)
        print(' *** NOTE: optional physics beyond upstream sitrack is ON:', physics)
    # small clouds are launch-bound: a whole chunk of records per launch (k_advect_multi, 4 us per record instead of
    # 11 us) and the rows of the chunk come back together; large clouds stream row by row
    small = world == 1 and physics is None and nP <= 262144 and nP * (Nt + 1) * 17 < 2e9 and not args.no_chunk
    deform = None
    if ndeform:
        # strain rates of buoy triangles, window by window on the GPU; the mesh is built from the seeds in the order the
        # files use (after --sort), so its vertices index the tracking file's `buoy` axis
        nwin = Nt // ndeform
        if nwin < 1:
            print('ERROR: --deform window (%d records) is longer than the run (%d records)!' % (ndeform, Nt))
            exit(0)
        tri = sit.TriangulateCloud(xPosC0, max_edge_km=args.deform_maxedge)
        if tri.shape[0] == 0:
            print('ERROR: --deform: no triangle left in the mesh of the buoys!')
            exit(0)
        print(' *** --deform: %d triangles, %d windows of %d records' % (tri.shape[0], nwin, ndeform))
        t1 = vTime[nwin * ndeform]
        dwriter = sit.DeformationWriter(nc_name('deformation', vTime[0], t1), nwin, tri, IDs, corigin=corgn)
        deform = dict(tri=tri, every=ndeform, sink=window_sink(ndeform, dwriter))
        if dscales:
            # boxes over the same mesh and seeds; only per-scale statistics leave the GPU
            H = sit.BoxHierarchy(xPosC0, tri, *dscales)
            print(' *** --deform-scales: %d levels of boxes from %g km, %s boxes' % (H.levels, H.L0_km, H.nbox.tolist()))
            swriter = sit.DeformationScalingWriter(nc_name('deformation-scaling', vTime[0], t1), nwin, H.scale_km,
                                                   H.bin_edges, corigin=corgn)
            deform.update(scales=H, scale_sink=window_sink(ndeform, swriter))
        if G is not None:
            # fixed cells over the model grid, membership rebuilt every window; only fields and statistics leave the GPU
            print(' *** --deform-grid: %d levels of cells from %g km, %d x %d level-1 cells from (%g, %g) km'
                  % (G.levels, G.L0_km, G.shape[0], G.shape[1], G.origin[0], G.origin[1]))
            gwriter = sit.DeformationGridWriter(nc_name('deformation-grid', vTime[0], t1), nwin, G, corigin=corgn)
            gswriter = sit.DeformationScalingWriter(nc_name('deformation-grid-scaling', vTime[0], t1), nwin,
                                                    G.scale_km, G.bin_edges, corigin=corgn)
            deform.update(grid=G, grid_sink=window_sink(ndeform, gwriter, gswriter))
        small = False                                             # windows close inside the streaming record loop
    dispersion = None
    if dspa:
        # pairs over the seeds in the order the files use (after --sort); only statistics leave the GPU
        nd, lags, npair, r_min, r_max = dspa
        nwd = Nt // nd
        pairs = sit.SeparationPairs(xPosC0, r_min, r_max, nP if npair is None else npair, seed=0)
        if pairs.shape[0] == 0:
            print('ERROR: --dispersion: no pair of distinct buoys was drawn!')
            exit(0)
        print(' *** --dispersion: %d pairs at %g to %g km, %d windows of %d records, lags 1..%d'
              % (pairs.shape[0], r_min, r_max, nwd, nd, lags))
        pwriter = sit.DispersionWriter(nc_name('dispersion', vTime[0], vTime[nwd * nd]), nwd,
                                       np.arange(1, lags + 1) * (nd * rdt / 86400.), sit.DEFAULT_R_EDGES,
                                       sit.DEFAULT_BIN_EDGES, corigin=corgn)
        dispersion = dict(pairs=pairs, every=nd, lags=lags, sink=window_sink(nd, pwriter))
        small = False
    fsle = None
    if fsla:
        # pairs over the seeds in the order the files use (after --sort), drawn as for --dispersion; the pairs' state
        # stays on the GPU and only statistics leave it
        nf, deltas, npair, r_min, r_max = fsla
        nwf = Nt // nf
        pairs = sit.SeparationPairs(xPosC0, r_min, r_max, nP if npair is None else npair, seed=0)
        if pairs.shape[0] == 0:
            print('ERROR: --fsle: no pair of distinct buoys was drawn!')
            exit(0)
        print(' *** --fsle: %d pairs at %g to %g km, %d thresholds from %g to %g km, %d samples of %d records'
              % (pairs.shape[0], r_min, r_max, deltas.size, deltas[0], deltas[-1], nwf, nf))
        fwriter = sit.FsleWriter(nc_name('fsle', vTime[0], vTime[nwf * nf]), nwf, deltas, sit.DEFAULT_TAU_EDGES,
                                 nf * rdt / 86400., corigin=corgn)
        fsle = dict(pairs=pairs, every=nf, deltas=deltas, sink=window_sink(nf, fwriter))
        small = False
    sample = None
    if smpa:
        # the SI3 fields along the trajectories, in the order the files use (after --sort); under torchrun each rank
        # samples its block and the samples travel to rank 0 with the rows
        snames, ns, sinterp = smpa
        nws = Nt // ns
        print(' *** --sample: %s (%s) at %d rows, every %d records' % (' '.join(snames), sinterp, nws + 1, ns))
        smwriter = None
        if rank == 0:
            smwriter = sit.SampleWriter(nc_name('sampled', vTime[0], vTime[Nt]), nws + 1, IDs, snames, sinterp, ns,
                                        units=sunits, corigin=corgn)
            writers.append(smwriter)

        def sample_sink(js, vals):
            if world == 1:
                smwriter.write(js, vTime[js * ns], vals)
            else:
                sample_stash.append((js, vals))
        sample = dict(names=snames, every=ns, interp=sinterp, tyx=(xYt, xXt), sink=sample_sink,
                      get=lambda k, n: ds.variables[n][k + kstrt, :, :])
        small = False                                             # rows are sampled inside the streaming record loop
    connect = None
    if cona:
        # the buoys' host cells against the region map, on the GPU; under torchrun each rank counts its block and the
        # windows' integer statistics are summed on rank 0 (every rank drains its windows in the same order)
        nc = cona[0]
        nwc = Nt // nc
        print(' *** --connect: %d regions of %s in %s, %d samples of %d records' % (nreg, cona[2], cona[1], nwc, nc))
        cwriter = None
        if rank == 0:
            cwriter = sit.ConnectivityWriter(nc_name('connectivity', vTime[0], vTime[nwc * nc]), nwc, nreg,
                                             sit.DEFAULT_TAU_EDGES, nc * rdt / 86400., corigin=corgn)
            writers.append(cwriter)

        def connect_sink(w, st):
            if world > 1:
                import torch
                t = torch.from_numpy(np.concatenate([np.ravel(st[k]) for k in sit.CONNECT_STATS]))
                dist.reduce(t, dst=0)
                if rank != 0:
                    return
                st = sit.connect.stats_dict(st['tau_edges'], st['sample_days'], st['nreg'], t.numpy())
            cwriter.write(w, vTime[w * nc], vTime[(w + 1) * nc], st)
        connect = dict(labels=labels, every=nc, sink=connect_sink)
        small = False                                             # windows close inside the streaming record loop
    if small:
        nchunk = max(2, min(Nt, 48, int(256e6 // (3 * Nj * Ni * 4))))      # <= 256 MB of pinned records per slot
        res = eng.track(record, Nt, kstrt=kstrt, pos0=xPosC0, posG0=xPosG0, rec_first=z1st, chunk=nchunk,
                        row_dtype=args.rows)
        for k in range(Nt):
            keep_row(k, res['posC'][k + 1], res['posG'][k + 1], res['mask'][k + 1])
    else:
        res = eng.track(record, Nt, kstrt=kstrt, rec_first=cut(z1st), sink=sink,
                        row_dtype='f8' if physics else args.rows, physics=physics, deform=deform,
                        dispersion=dispersion, fsle=fsle, sample=sample, connect=connect)
    eng.close()
    for w in writers:
        w.close()
    ds.close()
    n_alive = res['n_alive']
    if world > 1:
        import torch
        t = torch.from_numpy(np.ascontiguousarray(n_alive))
        dist.all_reduce(t)
        n_alive = t.numpy()
        dist.barrier()
        dist.destroy_process_group()
        if rank != 0:
            return 0
    if lUse2DTime:
        for jt in range(Nt):
            print('   *   record ' + str(jt + kstrt) + ': number of buoys alive = ' + str(int(n_alive[jt])))

    # ---- outputs (reference :498-571) ---------------------------------------------------------------
    if writer is not None:
        writer.close()
    if lUse2DTime:
        # per-buoy first and last valid rows; xTime follows from the windows (reference :334-340, :463)
        zTim = np.zeros((2, nP), dtype=int)
        zTim[0] = ztime_model[z1st] - int(rdt / 2)
        zTim[1] = np.where(zMSK[1] == 1, vTime[kN - 1] + int(rdt), int(sit.FillValue))
        zvt = np.array([np.mean(zTim[0, :]), np.mean(zTim[1, :])])
    else:
        zTim = []
        zvt = np.array([vTime[0], vTime[Nt]])
    sit.ncSaveCloudBuoys(nc_name('tracking12', zvt[0], zvt[1]), zvt, IDs, z2XY[:, :, 0], z2XY[:, :, 1], z2GC[:, :, 0],
                         z2GC[:, :, 1], mask=zMSK, xtime=zTim, corigin=corgn)
    print('        => global first and final dates in simulated trajectories:', e2c(zvt[0]), e2c(zvt[1]), '\n')
    return 0


if __name__ == '__main__':
    main()
