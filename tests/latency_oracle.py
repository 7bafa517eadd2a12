"""The oracle's restatement of a step with actuation latency (test support; not a test module).

`LatencyOracleEnv.step(action, latency)`: every command the controller issues is written `latency` substeps into its control period
(after the last substep when latency == frame_skip) and the previous command stays in force until then -- the engine's per-env
actuation latency (DESIGN.md section 10).  The controllers and the epilogue are OracleEnv.step's; each control period runs as
s.step(d), the commit, s.step(frame_skip - d).  With latency 0 it reproduces OracleEnv.step bit for bit (tests/test_latency.py)."""
import numpy as np

from oracle.oracle import OracleEnv, euler2quat, goal_distance, mju_mat2quat, mju_mulquat


class LatencyOracleEnv(OracleEnv):
    def _control_period(self, commit, latency):
        s = self.sim
        if latency > 0:
            s.step(latency)
        commit()
        if latency < self.frame_skip:
            s.step(self.frame_skip - latency)

    def step(self, action, latency=0):
        latency = int(latency)
        assert 0 <= latency <= self.frame_skip, latency
        action = np.clip(np.asarray(action, dtype=np.float32), np.float32(-1.0), np.float32(1.0))
        s = self.sim
        if self.controller_type == "IK":
            target_pos = s.site_xpos[self.site_eef] + action[:3] * np.float32(0.2)
            if self.fetch_env:
                target_quat = np.array([0, -0.707, 0, 0.707])
            else:
                quat_rot = euler2quat(action[3:6] * np.float32(0.5))
                target_quat = mju_mulquat(quat_rot, mju_mat2quat(s.site_xmat[self.site_eef]))
            ctrl_action = np.zeros(7)
            ctrl_action[-1] = 0.5 + np.float64(action[-1]) * 0.5
            for _ in range(self.control_steps):
                delta = self._ik_delta(target_pos, target_quat)       # from the frames and the ctrl in force at the block's start
                ctrl_action[:6] = s.ctrl[:6] + delta[:6]
                cmd = ctrl_action.copy()
                self._control_period(lambda: s.ctrl.__setitem__(slice(None), cmd), latency)
        elif self.controller_type == "mocap":
            tcp = self.flat["body_names"].index("gripper_tcp")
            mocap_action = np.zeros(7)
            mocap_action[:3] = action[:3] * np.float32(0.1)
            mocap_action[3:7] = np.array([0.5, -0.5, -0.5, 0.5]) if self.fetch_env else action[3:7]
            mocap_action[3:7] -= s.xquat[tcp]
            mpos = s.xpos[tcp] + mocap_action[:3]                     # computed at substep 0 from the stale frames
            mquat = s.xquat[tcp] + mocap_action[3:7]
            grip = 0.5 + np.float64(action[-1]) * 0.5

            def commit():
                s.mocap_pos[:] = mpos
                s.mocap_quat[:] = mquat
                s.ctrl[-1] = grip
            self._control_period(commit, latency)
        else:
            cmd = action.astype(np.float64)
            self._control_period(lambda: s.ctrl.__setitem__(slice(None), cmd), latency)
        if self.block_gripper:
            s.qpos[self.flat["jnt_qposadr"][self.j_rf]] = 0.0
            s.qpos[self.flat["jnt_qposadr"][self.j_lf]] = 0.0
            s.forward()
        obs = self._get_obs()
        d = goal_distance(self.achieved_goal, self.goal)
        is_success = bool(d < self.distance_threshold)
        reward = self.compute_reward(self.achieved_goal, self.goal, {})
        terminated = is_success
        self.elapsed += 1
        truncated = is_success or self.elapsed >= self.max_episode_steps
        return obs, reward, terminated, truncated, {"is_success": is_success}
