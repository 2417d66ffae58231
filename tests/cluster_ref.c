/*
 * cluster_ref.c — CPU reference of the clustering stage (include/mmw_radar.h: mmw_set_clustering).  Test infrastructure:
 * compiled by tests/cluster_ref.py into a temporary directory and loaded with ctypes; the library never links it.
 *
 * Parity status: UNPINNED by the reference program, which has no clustering stage.  This definition IS the specification;
 * it is cross-checked against scipy's connected components (tests/test_cluster_reference.py) and the GPU kernels
 * (csrc/mmw_cluster.cu) match it bit for bit (tests/test_gpu_clustering.py).  Plain C, fp64.
 *
 * Input: an ordered detection list (frame, range_bin, doppler_bin ascending: what the chain produces) of n_frames frames,
 * frame f holding dets[offsets[f] .. offsets[f+1]).  Within one frame, with the signed Doppler d' = d < Cp/2 ? d : d - Cp
 * (no wrap: a blob straddling +-Cp/2 is two objects), detections i and j are neighbours iff |r_i - r_j| <= eps_range,
 * |d'_i - d'_j| <= eps_doppler and |angle_bin_i - angle_bin_j| <= eps_angle.  Objects are the connected components with at
 * least min_points members (friends-of-friends: unique, no order-dependent border points), ordered by (frame, index of the
 * lowest-index member); at most max_objects_per_frame are kept per frame.
 * labels[i] (offsets[n_frames] entries): index of i's object in objs, or -1.  Sums are fp64 over the members in ascending
 * index, rounded to fp32 once; the products p*x are exact in fp64.
 * Returns the objects written (<= obj_cap); *n_total gets the true count, *flags bit 0 = some frame's objects were cut.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "mmw_radar.h"

/* ---- clustering: connected components of the neighbour graph of each frame ---- */
static int ref_signed_doppler(int d, int Cp) { return d < Cp / 2 ? d : d - Cp; }

typedef struct { double sp, sr, sd, sa; } ref_cluster_acc;

static long ref_uf_find(long *parent, long x)
{
    while (parent[x] != x) {
        parent[x] = parent[parent[x]];
        x = parent[x];
    }
    return x;
}

long ref_cluster(const mmw_detection *dets, const uint32_t *offsets, int n_frames, int Cp,
                 const mmw_cluster_params *cp, mmw_object *objs, long obj_cap, int32_t *labels,
                 long *n_total, uint32_t *flags)
{
    const long n = n_frames > 0 ? (long)offsets[n_frames] : 0;
    long *parent = (long *)malloc(sizeof(long) * (size_t)(n > 0 ? n : 1));
    long *size = (long *)calloc((size_t)(n > 0 ? n : 1), sizeof(long));
    long *obj_of_root = (long *)malloc(sizeof(long) * (size_t)(n > 0 ? n : 1));
    ref_cluster_acc *acc = (ref_cluster_acc *)calloc((size_t)(obj_cap > 0 ? obj_cap : 1), sizeof(ref_cluster_acc));
    long written = 0, total = 0;
    uint32_t fl = 0;
    for (long i = 0; i < n; ++i) { parent[i] = i; labels[i] = -1; obj_of_root[i] = -1; }
    for (int f = 0; f < n_frames; ++f) {
        const long s = offsets[f], e = offsets[f + 1];
        /* edges: every pair (j < i) of the frame within eps_range rows, found by walking back from i (the list is ordered by range) */
        for (long i = s; i < e; ++i) {
            const int ri = dets[i].range_bin, di = ref_signed_doppler(dets[i].doppler_bin, Cp), ai = dets[i].angle_bin;
            for (long j = i - 1; j >= s && ri - (int)dets[j].range_bin <= cp->eps_range; --j) {
                const int dj = ref_signed_doppler(dets[j].doppler_bin, Cp), aj = dets[j].angle_bin;
                if (abs(di - dj) > cp->eps_doppler || abs(ai - aj) > cp->eps_angle) continue;
                const long a = ref_uf_find(parent, i), b = ref_uf_find(parent, j);
                if (a < b) parent[b] = a;            /* the root of a component is its lowest index */
                else if (b < a) parent[a] = b;
            }
        }
        for (long i = s; i < e; ++i) size[ref_uf_find(parent, i)]++;
        /* objects in order of their lowest-index member */
        long k = 0;
        for (long i = s; i < e; ++i) {
            if (ref_uf_find(parent, i) != i || size[i] < cp->min_points) continue;
            ++total;
            if (k++ >= cp->max_objects_per_frame) { fl |= 1u; continue; }
            if (written < obj_cap) {
                mmw_object *o = &objs[written];
                memset(o, 0, sizeof(*o));
                o->frame = dets[i].frame;
                o->first_det = (uint32_t)i;
                obj_of_root[i] = written;
            }
            ++written;
        }
        /* labels: the object of the component, -1 for none or a cut one */
        for (long i = s; i < e; ++i) {
            const long r = ref_uf_find(parent, i);
            const long oi = obj_of_root[r];
            if (oi < 0) continue;
            labels[i] = (int32_t)oi;
        }
        /* one pass in ascending index: every object's sums run over its members in that order */
        for (long i = s; i < e; ++i) {
            const long oi = labels[i];
            if (oi < 0) continue;
            mmw_object *o = &objs[oi];
            ref_cluster_acc *a = &acc[oi];
            const double p = (double)dets[i].power;
            const int ds = ref_signed_doppler(dets[i].doppler_bin, Cp);
            if (o->n_det == 0) {
                o->peak_det = (uint32_t)i;
                o->range_min = o->range_max = dets[i].range_bin;
                o->doppler_min = o->doppler_max = (int16_t)ds;
            }
            a->sp += p;
            a->sr += p * (double)dets[i].range_bin;
            a->sd += p * (double)ds;
            a->sa += p * (double)dets[i].angle_rad;
            if (dets[i].power > dets[o->peak_det].power) o->peak_det = (uint32_t)i;   /* equal power: the lower index stays */
            if (dets[i].range_bin < o->range_min) o->range_min = dets[i].range_bin;
            if (dets[i].range_bin > o->range_max) o->range_max = dets[i].range_bin;
            if (ds < o->doppler_min) o->doppler_min = (int16_t)ds;
            if (ds > o->doppler_max) o->doppler_max = (int16_t)ds;
            o->n_det++;
        }
    }
    for (long oi = 0; oi < written && oi < obj_cap; ++oi) {
        mmw_object *o = &objs[oi];
        const ref_cluster_acc *a = &acc[oi];
        o->range_bin = a->sp > 0 ? (float)(a->sr / a->sp) : 0.f;
        o->doppler_bin = a->sp > 0 ? (float)(a->sd / a->sp) : 0.f;
        o->angle_rad = a->sp > 0 ? (float)(a->sa / a->sp) : 0.f;
        o->power = (float)a->sp;
        o->peak_power = dets[o->peak_det].power;
        o->peak_noise = dets[o->peak_det].noise;
    }
    free(acc);
    free(parent);
    free(size);
    free(obj_of_root);
    if (n_total) *n_total = total;
    if (flags) *flags = fl;
    return written < obj_cap ? written : obj_cap;
}
