/* rkfd_engine.h - batched device engine: B independent environments of one model, sharded over the
 * devices of one process in contiguous env blocks (no inter-device traffic on the step path,
 * SURVEY.md section 8e).  No CUDA type appears in this header. */
#ifndef RKFD_ENGINE_H
#define RKFD_ENGINE_H

#include <string>
#include <vector>

#include "rkfd_types.h"

namespace rkfd {

struct Shard;

class Engine {
 public:
  /* devices empty -> the current device */
  /* mp_default: the model's own mass properties of the declared links ([nmp][10], build_model), needed when model.nmp > 0 */
  Engine(const ModelDev &model, int B, const std::vector<int> &devices, const double *mp_default = nullptr);
  ~Engine();
  Engine(const Engine&) = delete;
  Engine &operator=(const Engine&) = delete;

  int B() const { return B_; }
  const ModelDev &model() const { return model_; }
  int num_shards() const { return (int)shards_.size(); }

  /* host arrays are env-major: q[B][nq], u[B][nl], contact arrays [B][nslot](x3) */
  void set_state(const double *q, const double *qd);
  void get_state(double *q, double *qd, double *qdd);
  void set_motor_input(const double *u);
  /* rows k0..k0+n-1 of q (which 0), q' (1) or the motor input (2) <- vals, for every environment (scalar setters on a running simulator) */
  void fill_rows(int which, int k0, int n, const double *vals);
  /* end-of-run statistics reduced on the device: sums [0] envs [1] envs in contact [2] active contact vertices [3] flagged envs; maxima [4] |q''| [5] |q'| */
  void stats(double out[8]);
  /* asynchronous variants (pinned host memory, valid until sync()); transfers overlap the step kernels */
  void set_state_async(const double *q, const double *qd);
  void set_motor_input_async(const double *u);
  void get_state_async(double *q, double *qd, double *qdd);
  void join();
  void get_pivot(int *type, double *prev_trq);
  void set_pivot(const int *type, const double *prev_trq);
  void get_contact(int *active, int *type, double *ref, double *f);
  void set_contact(const int *active, const int *type, const double *ref);
  void get_status(int *status);

  void eval(bool ref);        /* one dynamics evaluation on the committed state */
  void step(int nsteps);      /* rkFDUpdate x nsteps, asynchronous */
  void sync();

  /* single-shard only: run on a caller-owned stream (so that the caller's events bracket the kernels) */
  void set_stream(void *cuda_stream);
  /* device pointers of shard `s` (SoA [k][ld], see StateDev): 0 q, 1 qd, 2 qdd, 3 u */
  void *device_ptr(int s, int which, int *ld, int *B);
  /* environment re-sort (slots ordered by contact count every `steps` steps; 0: never - then slot = environment, which callers
   * of device_ptr need).  slot_map: perm[slot] = environment of shard s (host copy, B entries) */
  void set_resort_interval(int steps){ resort_interval_ = steps; }
  int resort_interval() const { return resort_interval_; }
  void slot_map(int s, int *perm);
  long long resorts() const;
  long long launches() const { return launches_; }
  long long resort_kernels() const { return resort_kernels_; }      /* kernels launched by the re-sorts (key, offsets, assign, row permutations, order) */

  /* environment reset: environments envs[0..n) of shard `shard` (local indices) restart from (q, q', u) - device arrays,
   * env-major [n][nq] / [n][nl] - with every other per-environment row as a new engine holds it, and the committing
   * evaluation of rkFDUpdateInit runs for them alone.  qd null: zero, u null: the current input.  Entries outside [0, B) are
   * skipped; duplicates leave the environment with one of their states.  Stream-ordered on the shard's stream (the first
   * call, and a call with a longer list than any before, allocates and synchronises the device) */
  void reset_envs(int shard, int n, const int *envs, const double *q, const double *qd, const double *u);
  /* the same from host arrays, global environment indices (in range, no duplicates: the caller checks); synchronous */
  void reset_envs_host(int n, const int *envs, const double *q, const double *qd, const double *u);
  long long reset_kernels() const { return reset_kernels_; }        /* gather, zero fill and scatter launches of the resets */

  /* external wrench of the declared links (ModelDev::nfext), env-major [B][nfext][6]: (force, torque about the centre of mass),
   * world axes.  set_ext_wrench: host array, global environment index, every shard; synchronous.  set_ext_wrench_device: a
   * device buffer [Bs][nfext][6] of shard `shard`, indexed by the environment local to the shard, read through the slot
   * permutation by the transposing scatter; stream-ordered on the shard's stream, no allocation.  Both throw without a
   * declared link */
  void set_ext_wrench(const double *w);
  void set_ext_wrench_device(int shard, const double *w);
  /* mass properties of the declared links (ModelDev::nmp), env-major [B][nmp][10]: (mass, centre of mass, inertia about the
   * centre of mass xx xy xz yy yz zz), link axes.  set_mass_prop: host array, every shard, synchronous.  set_mass_prop_device:
   * a device buffer [Bs][nmp][10] of shard `shard`, indexed by the environment local to the shard; stream-ordered, no
   * allocation.  Both throw without a declared link; neither checks the values */
  void set_mass_prop(const double *mp);
  void set_mass_prop_device(int shard, const double *mp);

  /* link kinematics (rkfd_kin.cuh): world frames [B][nsel][12] (R row-major, p) and velocities [B][nsel][6] (linear, angular;
   * world axes) of the output columns of table `t`, from the committed state; a null output is neither computed nor written.
   * Nothing of the engine's state is written.  link_frames: device buffers of shard `shard`, indexed by the environment local
   * to the shard; stream-ordered on the shard's stream, no allocation.  link_frames_host: host arrays, global environment
   * index, every shard; synchronous */
  void link_frames(int shard, const KinDev &t, double *frame, double *vel);
  void link_frames_host(const KinDev &t, double *frame, double *vel);
  long long link_frame_kernels() const { return kin_kernels_; }     /* kinematics launches (one per shard and call) */

  /* net contact wrench [B][nsel][6] (force, torque about the link origin; world axes) of the last committing evaluation on the
   * output columns of table `t` (rkfd_link_contact.cuh), from the committed q and the contact forces.  Nothing of the engine's
   * state is written.  link_contact_wrench: a device buffer of shard `shard`, indexed by the environment local to the shard;
   * stream-ordered on the shard's stream, no allocation.  link_contact_wrench_host: a host array, global environment index,
   * every shard; synchronous */
  void link_contact_wrench(int shard, const LcwDev &t, double *w);
  void link_contact_wrench_host(const LcwDev &t, double *w);
  long long link_contact_kernels() const { return lcw_kernels_; }   /* launches (one per shard and call) */

  /* the step-kernel variant shard `shard` launches: v = (block, gscr, rigid, spec, minb); throws on a bad shard index */
  void kernel_variant(int shard, int v[5]) const;

 private:
  void upload_model(Shard &s);
  void launch(Shard &s, const StateDev &st, int cur, int mode, int nsteps);
  void resort(Shard &s);
  void reset_chunk(Shard &s, int n, const int *envs, const double *q, const double *qd, const double *u);
  void kin_launch(Shard &s, const KinDev &t, double *frame, double *vel);
  void lcw_launch(Shard &s, const LcwDev &t, double *w);
  int resort_interval_ = 0;
  ModelDev model_, model_tm_;     /* model_tm_: the same table with the tensor-memory scratch map (generic TM kernel) */
  int B_;
  std::vector<Shard*> shards_;
  long long launches_ = 0, resort_kernels_ = 0, reset_kernels_ = 0, kin_kernels_ = 0, lcw_kernels_ = 0;
  int id_;
};

/* throws std::runtime_error with the CUDA error string */
void cuda_check(int err, const char *what);
int device_count();
/* sustained fp64 FMA throughput of the current device, TFLOP/s (register-resident DFMA loop on all SMs) */
double measure_fp64_tflops();

}  // namespace rkfd
#endif
