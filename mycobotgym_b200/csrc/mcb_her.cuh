// Device-resident hindsight-experience replay ("future" strategy) -- SURVEY 8 f4, the caller on the far side of the step:
// mycobotgym/scripts/train.py:89-97 builds stable_baselines3.HerReplayBuffer(n_sampled_goal=4, goal_selection_strategy=
// "future") around the env and the buffer calls env.compute_reward on relabelled goals (mycobot.py:289-295).  The ring,
// the episode table (ep_start / ep_length per stored transition, stable_baselines3==2.0.0a0 her_replay_buffer.py) and
// the relabelling gather live in HBM so a rollout of 16 K envs never leaves the device.  Included by mcb_engine.cu.
//
// Layout: time-major rings [T][N][.] -- one add() writes N contiguous rows per array (coalesced D2D copies), a sample
// gathers single rows (obs_dim doubles = 80..200 B; one lane draws one sample, the warp copies its 32 rows).  HBM-bound:
// (2*obs_dim + 9) doubles + action floats read and written per sample.

struct mcb_her {
  int n_envs, T, obs_dim, action_dim, reward_type, n_sampled_goal, device;
  double thr;
  uint64_t seed;
  int pos, full;
  unsigned long long draws;            // sample() calls so far: part of the Philox counter
  double *obs, *next_obs, *ag, *next_ag, *dg;
  float *actions, *rewards;
  uint8_t *dones, *timeouts;
  int *ep_start, *ep_length, *cur_start;
  long long* n_valid;                  // device counter: transitions that belong to complete, not yet overwritten episodes
};

namespace {

// add(), step 1: the slot about to be overwritten may belong to a stored episode -> the rest of that episode is
// invalidated (ep_length := 0), then the slot is tagged with the running episode's start.
__global__ void her_invalidate_kernel(int* ep_start, int* ep_length, const int* cur_start, long long* n_valid, int N, int T, int pos) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  int es = ep_start[(size_t)pos * N + i], el = ep_length[(size_t)pos * N + i];
  if (el > 0) {
    int end = es + el, cnt = 0;
    for (int t = pos; t < end && cnt < T; t++, cnt++) ep_length[(size_t)(t % T) * N + i] = 0;
    atomicAdd((unsigned long long*)n_valid, (unsigned long long)(-(long long)cnt));
  }
  ep_start[(size_t)pos * N + i] = cur_start[i];
}

// add(), step 2 (after pos advanced to pos_new): envs whose episode just ended get ep_length filled in for every
// transition of that episode (_compute_episode_length) and start a new episode at pos_new.
__global__ void her_close_episode_kernel(int* ep_length, int* cur_start, const uint8_t* dones, long long* n_valid, int N, int T, int pos_new) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N || !dones[i]) return;
  int start = cur_start[i], end = pos_new;
  if (end < start) end += T;
  for (int t = start; t < end; t++) ep_length[(size_t)(t % T) * N + i] = end - start;
  atomicAdd((unsigned long long*)n_valid, (unsigned long long)(end - start));
  cur_start[i] = pos_new;
}

__global__ void f64_to_f32_kernel(const double* in, float* out, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (float)in[i];
}

__global__ void her_flags_kernel(uint8_t* dones, uint8_t* timeouts, const uint8_t* term, const uint8_t* trunc, int N) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  uint8_t te = term[i] != 0, tr = trunc[i] != 0;
  dones[i] = te | tr;                 // VecEnv: done = terminated or truncated
  timeouts[i] = tr & !te;             // info["TimeLimit.truncated"] = truncated and not terminated
}

struct HerSampleArgs {
  const double *obs, *next_obs, *ag, *next_ag, *dg;
  const float *actions, *rewards;
  const uint8_t *dones, *timeouts;
  const int *ep_start, *ep_length;
  int N, T, od, ad, size, batch, nb_virtual, reward_type;
  double thr;
  uint64_t seed;
  unsigned long long draw0;
  const int64_t* inj_index;            // [batch] flat index t * N + env, or null: drawn on the device
  const int32_t* inj_future;           // [batch] transition index inside the episode for the virtual samples, or null
  double *o_obs, *o_ag, *o_dg, *o_next_obs, *o_next_ag;
  float *o_actions, *o_rewards, *o_dones;
  int64_t* o_index;                    // optional: (flat index, relabel source flat index or -1) per sample
  int* o_fail;
};

// One lane draws one sample (index, and for the virtual ones the relabel source), then the warp copies its 32 rows
// cooperatively, eight rows in flight at a time: the gather is a stream of independent 200-byte reads from random places of
// the ring, so memory-level parallelism -- not the copy width -- is what the kernel needs.
__global__ void __launch_bounds__(128) her_sample_kernel(HerSampleArgs a) {
  const int lane = threadIdx.x & 31;
  const int b = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32 + lane;
  const int b0 = b - lane;
  if (b0 >= a.batch) return;
  int t = 0, env = 0, src = -1;
  if (b < a.batch) {
    unsigned long long ctr = a.draw0 * 4096ull;
    bool ok = true;
    if (a.inj_index) { t = (int)(a.inj_index[b] / a.N); env = (int)(a.inj_index[b] % a.N); ok = a.ep_length[(size_t)t * a.N + env] > 0; }
    else {
      // uniform over the transitions of complete episodes == np.random.choice(np.flatnonzero(ep_length > 0)): rejection
      int guard = 0;
      do {
        t = min(a.size - 1, (int)(philox_uniform(a.seed, (uint32_t)b, ctr) * a.size));
        env = min(a.N - 1, (int)(philox_uniform(a.seed, (uint32_t)b, ctr) * a.N));
      } while (a.ep_length[(size_t)t * a.N + env] <= 0 && ++guard < 2000);
      ok = a.ep_length[(size_t)t * a.N + env] > 0;
    }
    if (!ok) { atomicAdd(a.o_fail, 1); t = 0; env = 0; }
    else if (b < a.nb_virtual) {
      // _sample_goals, strategy "future": a transition of the same episode at or after the current one
      int es = a.ep_start[(size_t)t * a.N + env], el = a.ep_length[(size_t)t * a.N + env];
      int cur = ((t - es) % a.T + a.T) % a.T;
      int fut;
      if (a.inj_future) fut = a.inj_future[b];
      else fut = min(el - 1, cur + (int)(philox_uniform(a.seed, (uint32_t)b, ctr) * (el - cur)));      // np.random.randint(cur, el)
      src = (fut + es) % a.T;
    }
    const size_t row = (size_t)t * a.N + env;
    // per-sample scalars: goal, reward, done (this lane's own sample)
    double nag[3], g[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
      nag[k] = a.next_ag[row * 3 + k];
      g[k] = src >= 0 ? a.next_ag[((size_t)src * a.N + env) * 3 + k] : a.dg[row * 3 + k];
      a.o_ag[(size_t)b * 3 + k] = a.ag[row * 3 + k];
      a.o_next_ag[(size_t)b * 3 + k] = nag[k];
      a.o_dg[(size_t)b * 3 + k] = g[k];
    }
    float r;
    if (src >= 0) {
      // compute_reward(next_achieved_goal, new_goal) (mycobot.py:289-295), stored as float32 like SB3's reward array
      const double dx = nag[0] - g[0], dy = nag[1] - g[1], dz = nag[2] - g[2];
      const double d = sqrt(dx * dx + dy * dy + dz * dz);
      r = a.reward_type == 0 ? -(float)(d > a.thr) : (float)(-d);
    } else r = a.rewards[row];
    a.o_rewards[b] = r;
    a.o_dones[b] = (float)(a.dones[row] * (1 - a.timeouts[row]));
    if (a.o_index) { a.o_index[2 * (size_t)b] = (int64_t)row; a.o_index[2 * (size_t)b + 1] = src >= 0 ? (int64_t)src * a.N + env : -1; }
  }
  // cooperative row copies: observation, next observation, action of samples b0 .. b0 + 31
  const long long myrow = (b < a.batch) ? (long long)t * a.N + env : -1;
#pragma unroll 1
  for (int k0 = 0; k0 < 32; k0 += 8) {
    long long rows[8];
#pragma unroll
    for (int u = 0; u < 8; u++) rows[u] = __shfl_sync(FULLMASK, myrow, k0 + u);
    for (int c = lane; c < a.od; c += 32) {
      double vo[8], vn[8];
#pragma unroll
      for (int u = 0; u < 8; u++) if (rows[u] >= 0) { vo[u] = a.obs[(size_t)rows[u] * a.od + c]; vn[u] = a.next_obs[(size_t)rows[u] * a.od + c]; }
#pragma unroll
      for (int u = 0; u < 8; u++) if (rows[u] >= 0) { a.o_obs[(size_t)(b0 + k0 + u) * a.od + c] = vo[u]; a.o_next_obs[(size_t)(b0 + k0 + u) * a.od + c] = vn[u]; }
    }
    if (lane < a.ad) {
      float va[8];
#pragma unroll
      for (int u = 0; u < 8; u++) if (rows[u] >= 0) va[u] = a.actions[(size_t)rows[u] * a.ad + lane];
#pragma unroll
      for (int u = 0; u < 8; u++) if (rows[u] >= 0) a.o_actions[(size_t)(b0 + k0 + u) * a.ad + lane] = va[u];
    }
  }
}

}  // namespace

extern "C" {

int32_t mcb_her_create(int32_t n_envs, int32_t buffer_steps, int32_t obs_dim, int32_t action_dim, int32_t n_sampled_goal,
                       int32_t reward_type, double distance_threshold, uint64_t seed, mcb_her** out) {
  if (!out || n_envs <= 0 || buffer_steps <= 1 || obs_dim <= 0 || action_dim <= 0 || n_sampled_goal < 0) return fail("mcb_her_create: bad argument");
  if (reward_type != 0 && reward_type != 1) return fail("mcb_her_create: relabelled rewards exist for the sparse and dense rewards only (reward_shaping needs the simulation state)");
  mcb_her* h = new mcb_her();
  memset(h, 0, sizeof(*h));
  h->n_envs = n_envs; h->T = buffer_steps; h->obs_dim = obs_dim; h->action_dim = action_dim; h->reward_type = reward_type;
  h->n_sampled_goal = n_sampled_goal; h->thr = distance_threshold; h->seed = seed;
  cudaGetDevice(&h->device);
  const size_t R = (size_t)n_envs * buffer_steps;
  // partial allocations are released on failure (mcb_her_destroy frees whatever is non-null)
#define HCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { mcb_her_destroy(h); return fail("mcb_her_create: " #call, e_); } } while (0)
#define HALLOC(p, n) HCK(cudaMalloc(&(p), (n)))
  HALLOC(h->obs, R * obs_dim * sizeof(double)); HALLOC(h->next_obs, R * obs_dim * sizeof(double));
  HALLOC(h->ag, R * 3 * sizeof(double)); HALLOC(h->next_ag, R * 3 * sizeof(double)); HALLOC(h->dg, R * 3 * sizeof(double));
  HALLOC(h->actions, R * action_dim * sizeof(float)); HALLOC(h->rewards, R * sizeof(float));
  HALLOC(h->dones, R); HALLOC(h->timeouts, R);
  HALLOC(h->ep_start, R * sizeof(int)); HALLOC(h->ep_length, R * sizeof(int)); HALLOC(h->cur_start, n_envs * sizeof(int));
  HALLOC(h->n_valid, sizeof(long long));
  HCK(cudaMemset(h->ep_start, 0, R * sizeof(int))); HCK(cudaMemset(h->ep_length, 0, R * sizeof(int)));
  HCK(cudaMemset(h->cur_start, 0, n_envs * sizeof(int))); HCK(cudaMemset(h->n_valid, 0, sizeof(long long)));
#undef HALLOC
#undef HCK
  *out = h;
  return 0;
}

void mcb_her_destroy(mcb_her* h) {
  if (!h) return;
  cudaFree(h->obs); cudaFree(h->next_obs); cudaFree(h->ag); cudaFree(h->next_ag); cudaFree(h->dg); cudaFree(h->actions);
  cudaFree(h->rewards); cudaFree(h->dones); cudaFree(h->timeouts); cudaFree(h->ep_start); cudaFree(h->ep_length);
  cudaFree(h->cur_start); cudaFree(h->n_valid);
  delete h;
}

int32_t mcb_her_add(mcb_her* h, const double* obs, const double* achieved_goal, const double* desired_goal, const double* next_obs,
                    const double* next_achieved_goal, const float* actions, const void* rewards, int32_t rewards_f64,
                    const uint8_t* terminated, const uint8_t* truncated, void* stream) {
  if (!h || !obs || !achieved_goal || !desired_goal || !next_obs || !next_achieved_goal || !actions || !rewards || !terminated || !truncated)
    return fail("mcb_her_add: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int N = h->n_envs, T = h->T, pos = h->pos;
  const size_t od = h->obs_dim, ad = h->action_dim, base = (size_t)pos * N;
  const unsigned grid = (N + 255) / 256;
  her_invalidate_kernel<<<grid, 256, 0, st>>>(h->ep_start, h->ep_length, h->cur_start, h->n_valid, N, T, pos);
  CK(cudaMemcpyAsync(h->obs + base * od, obs, N * od * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(h->next_obs + base * od, next_obs, N * od * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(h->ag + base * 3, achieved_goal, N * 3 * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(h->next_ag + base * 3, next_achieved_goal, N * 3 * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(h->dg + base * 3, desired_goal, N * 3 * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(h->actions + base * ad, actions, N * ad * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (rewards_f64) f64_to_f32_kernel<<<grid, 256, 0, st>>>((const double*)rewards, h->rewards + base, N);
  else CK(cudaMemcpyAsync(h->rewards + base, rewards, N * sizeof(float), cudaMemcpyDeviceToDevice, st));
  her_flags_kernel<<<grid, 256, 0, st>>>(h->dones + base, h->timeouts + base, terminated, truncated, N);
  const int pos_new = (pos + 1) % T;
  her_close_episode_kernel<<<grid, 256, 0, st>>>(h->ep_length, h->cur_start, h->dones + base, h->n_valid, N, T, pos_new);
  CK(cudaGetLastError());
  h->pos = pos_new;
  if (pos_new == 0) h->full = 1;
  return 0;
}

int64_t mcb_her_size(const mcb_her* h) { return h ? (int64_t)(h->full ? h->T : h->pos) * h->n_envs : -1; }

int32_t mcb_her_episode_table(mcb_her* h, int32_t* ep_start, int32_t* ep_length, int64_t* n_valid, void* stream) {
  if (!h) return fail("mcb_her_episode_table: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t R = (size_t)h->n_envs * h->T;
  if (ep_start) CK(cudaMemcpyAsync(ep_start, h->ep_start, R * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (ep_length) CK(cudaMemcpyAsync(ep_length, h->ep_length, R * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (n_valid) { CK(cudaMemcpyAsync(n_valid, h->n_valid, sizeof(long long), cudaMemcpyDeviceToHost, st)); CK(cudaStreamSynchronize(st)); }
  return 0;
}

int32_t mcb_her_sample(mcb_her* h, int32_t batch_size, const int64_t* inj_index, const int32_t* inj_future, double* obs, double* achieved_goal,
                       double* desired_goal, double* next_obs, double* next_achieved_goal, float* actions, float* rewards, float* dones,
                       int64_t* index_out, int32_t* fail_count, void* stream) {
  if (!h || batch_size <= 0 || !obs || !achieved_goal || !desired_goal || !next_obs || !next_achieved_goal || !actions || !rewards || !dones || !fail_count)
    return fail("mcb_her_sample: bad argument");
  const int size = h->full ? h->T : h->pos;
  if (size == 0) return fail("mcb_her_sample: the buffer is empty");
  cudaStream_t st = (cudaStream_t)stream;
  HerSampleArgs a;
  a.obs = h->obs; a.next_obs = h->next_obs; a.ag = h->ag; a.next_ag = h->next_ag; a.dg = h->dg; a.actions = h->actions; a.rewards = h->rewards;
  a.dones = h->dones; a.timeouts = h->timeouts; a.ep_start = h->ep_start; a.ep_length = h->ep_length;
  a.N = h->n_envs; a.T = h->T; a.od = h->obs_dim; a.ad = h->action_dim; a.size = size; a.batch = batch_size;
  // her_ratio = 1 - 1 / (n_sampled_goal + 1); the first int(her_ratio * batch) samples are virtual (relabelled)
  const double her_ratio = 1.0 - 1.0 / (double)(h->n_sampled_goal + 1);
  a.nb_virtual = (int)(her_ratio * (double)batch_size);
  a.reward_type = h->reward_type; a.thr = h->thr; a.seed = h->seed ^ 0x48455221ull; a.draw0 = h->draws++;
  a.inj_index = inj_index; a.inj_future = inj_future;
  a.o_obs = obs; a.o_ag = achieved_goal; a.o_dg = desired_goal; a.o_next_obs = next_obs; a.o_next_ag = next_achieved_goal;
  a.o_actions = actions; a.o_rewards = rewards; a.o_dones = dones; a.o_index = index_out; a.o_fail = fail_count;
  CK(cudaMemsetAsync(fail_count, 0, sizeof(int), st));
  her_sample_kernel<<<(batch_size + 127) / 128, 128, 0, st>>>(a);
  CK(cudaGetLastError());
  return 0;
}

}  // extern "C"
