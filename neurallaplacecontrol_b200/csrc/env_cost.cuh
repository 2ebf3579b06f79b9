// Running cost of the three delayed ODE-RL environments:
//   running_cost(state, u) = -(diff_obs_reward_(state, exp_reward=False) + diff_ac_reward_(u))
// (closure mppi_with_model.py:145-171; rewards envs/oderl/envs/ctpendulum.py:139-155,
// ctcartpole.py:289-346, ctacrobot.py:153-166,233-255, base_env.py:28-29,297-301), and one Euler step of
// the analytic delayed dynamics (oracle.py:11-224) for the NLC_DYN_ANALYTIC_DELAY slot.
#pragma once
#include "common.cuh"

namespace nlc {

__device__ __forceinline__ float trig2angle(float c, float s) {  // base_env.py:297-301
  const float C = c * c + s * s;
  c = c / C; s = s / C;
  return atan2f(s / C, c / C);
}

__device__ __forceinline__ float env_running_cost(const nlc_rollout_opts& o, const float* s, const float* u, int nu) {
  float ac = 0.0f;
  for (int i = 0; i < nu; ++i) ac = fmaf(u[i], u[i], ac);
  if (o.env == NLC_ENV_PENDULUM) {
    const float om = 1.0f - s[0];
    const float state_reward = -(om * om + s[1] * s[1]);
    const float reward = state_reward + 0.01f * (-(s[2] * s[2])) + (-0.01f * ac);
    return -reward;
  } else if (o.env == NLC_ENV_CARTPOLE) {
    const float ex = (s[0] + s[3]) - o.goal_x;  // ee_pos = (x + sin*l, cos*l), goal (goal_x, l), l = 1
    const float ey = s[2] - 1.0f;
    float state_reward;
    if (o.state_constraint) state_reward = -((ex * ex + expf(ex * 10.0f + 7.0f)) + ey * ey);
    else state_reward = -(ex * ex + ey * ey);
    const float vel = -(s[1] * s[1]) - s[4] * s[4];
    const float reward = state_reward + 0.01f * vel + (-0.01f * ac);
    return -reward;
  } else {
    const float th1 = trig2angle(s[0], s[1]);
    const float th2 = trig2angle(s[2], s[3]);
    const float vel = -(s[4] * s[4]) - s[5] * s[5];
    float s1, c1, s12, c12;
    sincosf(th1, &s1, &c1);
    sincosf(th1 + th2, &s12, &c12);
    const float p2x = -c1 - c12, p2y = s1 + s12;
    const float dx = p2x - 2.0f;
    const float state_reward = -(dx * dx) - p2y * p2y;
    const float reward = state_reward + 0.1f * vel + (-1e-4f * ac);
    return -reward;
  }
}

// Same cost for the tensor-core rollout (rollout_tc2.cu), where the acrobot's atan2 -> sincos round trip
// (ctacrobot.py:153-166,233-255) sat on the critical path of every step: cos(atan2(s, c)) = c / sqrt(c^2 + s^2), so the
// angles are never formed - an algebraic identity (difference ~1 ulp of fp32), pendulum and cartpole unchanged.
__device__ __forceinline__ float env_running_cost_fast(const nlc_rollout_opts& o, const float* s, const float* u, int nu) {
  // (pendulum and cartpole restated here rather than calling env_running_cost: its acrobot branch - atan2f and two sincosf
  // with their slow paths, ~480 instructions - would be compiled into every call site of the rollout's step loop)
  float ac = 0.0f;
  for (int i = 0; i < nu; ++i) ac = fmaf(u[i], u[i], ac);
  if (o.env == NLC_ENV_PENDULUM) {
    const float om = 1.0f - s[0];
    const float state_reward = -(om * om + s[1] * s[1]);
    return -(state_reward + 0.01f * (-(s[2] * s[2])) + (-0.01f * ac));
  }
  if (o.env == NLC_ENV_CARTPOLE) {
    const float ex = (s[0] + s[3]) - o.goal_x, ey = s[2] - 1.0f;
    float state_reward;
    if (o.state_constraint) state_reward = -((ex * ex + expf(ex * 10.0f + 7.0f)) + ey * ey);
    else state_reward = -(ex * ex + ey * ey);
    const float vel = -(s[1] * s[1]) - s[4] * s[4];
    return -(state_reward + 0.01f * vel + (-0.01f * ac));
  }
  const float r1 = rsqrtf(fmaf(s[0], s[0], s[1] * s[1])), r2 = rsqrtf(fmaf(s[2], s[2], s[3] * s[3]));
  const float c1 = s[0] * r1, s1 = s[1] * r1, c2 = s[2] * r2, s2 = s[3] * r2;
  const float c12 = fmaf(c1, c2, -(s1 * s2)), s12 = fmaf(s1, c2, c1 * s2);
  const float vel = -(s[4] * s[4]) - s[5] * s[5];
  const float p2x = -c1 - c12, p2y = s1 + s12;
  const float dx = p2x - 2.0f;
  const float state_reward = -(dx * dx) - p2y * p2y;
  const float reward = state_reward + 0.1f * vel + (-1e-4f * ac);
  return -reward;
}

// One explicit-Euler step with the action delayed by `delay` entries (oracle.py:11-224, friction=False,
// trigonometric observation form).  `u` points at window[-(delay+1)].
__device__ __forceinline__ void env_analytic_step(const nlc_rollout_opts& o, float* s, const float* u) {
  const float ts = o.dt;
  if (o.env == NLC_ENV_PENDULUM) {
    const float th = trig2angle(s[0], s[1]);
    const float thdot = s[2];
    const float uu = fminf(fmaxf(u[0], -2.0f), 2.0f);
    const float newth = th + thdot * ts;
    float sn, cs;
    sincosf(newth, &sn, &cs);
    const float newthdot = thdot + (-15.0f * sinf(th + 3.14159265358979f) + 3.0f * uu) * ts;
    s[0] = cs; s[1] = sn; s[2] = newthdot;
  } else if (o.env == NLC_ENV_CARTPOLE) {
    const float x = s[0], x_dot = s[1], theta_dot = s[4];
    const float C = s[2] * s[2] + s[3] * s[3];
    const float costheta = s[2] / C, sintheta = s[3] / C;
    const float theta = atan2f(sintheta / C, costheta / C);
    const float gravity = 9.8f, force_mag = 3.0f, masspole = 0.1f, total_mass = 1.1f, polemass_length = 0.1f;
    const float uu = fminf(fmaxf(u[0], -3.0f), 3.0f);
    const float force = uu * force_mag;
    const float temp = (force + polemass_length * theta_dot * theta_dot * sintheta) / total_mass;
    const float thetaacc = (gravity * sintheta - costheta * temp) / (1.0f * (4.0f / 3.0f - masspole * costheta * costheta / total_mass));
    const float xacc = temp - polemass_length * thetaacc * costheta / total_mass;
    const float new_theta = theta + theta_dot * ts;
    float sn, cs;
    sincosf(new_theta, &sn, &cs);
    s[0] = x + x_dot * ts; s[1] = x_dot + xacc * ts; s[2] = cs; s[3] = sn; s[4] = theta_dot + thetaacc * ts;
  } else {
    const float theta1 = trig2angle(s[0], s[1]);
    const float theta2 = trig2angle(s[2], s[3]);
    const float dtheta1 = s[4], dtheta2 = s[5];
    const float g = 9.8f, half_pi = 1.57079632679489662f;
    const float u0 = fminf(fmaxf(u[0], -5.0f), 5.0f), u1 = fminf(fmaxf(u[1], -5.0f), 5.0f);
    const float c2 = cosf(theta2), s2 = sinf(theta2);
    // m1=m2=1, l1=1, lc1=lc2=0.5, I1=I2=1
    const float d1 = 0.25f + (1.0f + 0.25f + c2) + 1.0f + 1.0f;
    const float d2 = (0.25f + 0.5f * c2) + 1.0f;
    const float phi2 = 0.5f * g * cosf(theta1 + theta2 - half_pi);
    const float phi1 = -0.5f * dtheta2 * dtheta2 * s2 - dtheta2 * dtheta1 * s2 + 1.5f * g * cosf(theta1 - half_pi) + phi2;
    const float ddtheta2 = (u0 + d2 / d1 * phi1 - 0.5f * dtheta1 * dtheta1 * s2 - phi2) / (0.25f + 1.0f - d2 * d2 / d1);
    const float ddtheta1 = -(u1 + d2 * ddtheta2 + phi1) / d1;
    const float nt1 = theta1 + dtheta1 * ts, nt2 = theta2 + dtheta2 * ts;
    float sa, ca, sb, cb;
    sincosf(nt1, &sa, &ca);
    sincosf(nt2, &sb, &cb);
    s[0] = ca; s[1] = sa; s[2] = cb; s[3] = sb; s[4] = dtheta1 + ddtheta1 * ts; s[5] = dtheta2 + ddtheta2 * ts;
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// fp64 forms for the fp64 planner (planner_f64.cu, model_grad.cu plan_f64_rollout_kernel): the reference's expressions in
// its own evaluation order (oracle/costs.py, oracle/dynamics.py), acrobot through atan2 / sincos as the reference does.
// goal_x and dt come in fp64 (the float opts cannot hold dt = 0.05 exactly).
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double trig2angle(double c, double s) {  // base_env.py:297-301
  const double C = c * c + s * s;
  c = c / C; s = s / C;
  return atan2(s / C, c / C);
}

__device__ __forceinline__ double env_running_cost(int env, int state_constraint, double goal_x, const double* s, const double* u,
                                                   int nu) {
  double ac = 0.0;
  for (int i = 0; i < nu; ++i) ac = ac + u[i] * u[i];
  if (env == NLC_ENV_PENDULUM) {
    const double om = 1.0 - s[0];
    const double state_reward = -(om * om + s[1] * s[1]);
    const double reward = state_reward + 0.01 * (-(s[2] * s[2]));
    return -(reward + (-0.01 * ac));
  } else if (env == NLC_ENV_CARTPOLE) {
    const double ex = (s[0] + s[3]) - goal_x;
    const double ey = s[2] - 1.0;
    const double state_reward = state_constraint ? -((ex * ex + exp(ex * 10.0 + 7.0)) + ey * ey) : -(ex * ex + ey * ey);
    const double vel = -(s[1] * s[1]) - s[4] * s[4];
    const double reward = state_reward + 0.01 * vel;
    return -(reward + (-0.01 * ac));
  } else {
    const double th1 = trig2angle(s[0], s[1]);
    const double th2 = trig2angle(s[2], s[3]);
    const double vel = -(s[4] * s[4]) - s[5] * s[5];
    double s1, c1, s12, c12;
    sincos(th1, &s1, &c1);
    sincos(th1 + th2, &s12, &c12);
    const double p2x = -c1 - c12, p2y = s1 + s12;
    const double dx = (p2x - 1.0) - 1.0;
    const double state_reward = -(dx * dx) - p2y * p2y;
    const double reward = state_reward + 0.1 * vel;
    return -(reward + (-1e-4 * ac));
  }
}

__device__ __forceinline__ void env_analytic_step(int env, double ts, double* s, const double* u) {
  if (env == NLC_ENV_PENDULUM) {
    const double th = trig2angle(s[0], s[1]);
    const double thdot = s[2];
    const double uu = fmin(fmax(u[0], -2.0), 2.0);
    const double newth = th + thdot * ts;
    const double newthdot = thdot + (-15.0 * sin(th + 3.141592653589793) + 3.0 * uu) * ts;
    double sn, cs;
    sincos(newth, &sn, &cs);
    s[0] = cs; s[1] = sn; s[2] = newthdot;
  } else if (env == NLC_ENV_CARTPOLE) {
    const double x = s[0], x_dot = s[1], theta_dot = s[4];
    const double C = s[2] * s[2] + s[3] * s[3];
    const double costheta = s[2] / C, sintheta = s[3] / C;
    const double theta = atan2(sintheta / C, costheta / C);
    const double force = fmin(fmax(u[0], -3.0), 3.0) * 3.0;
    const double total_mass = 0.1 + 1.0, pml = 0.1 * 1.0;
    const double temp = (force + pml * theta_dot * theta_dot * sintheta) / total_mass;
    const double thetaacc = (9.8 * sintheta - costheta * temp) / (1.0 * (4.0 / 3.0 - 0.1 * costheta * costheta / total_mass));
    const double xacc = temp - pml * thetaacc * costheta / total_mass;
    const double new_theta = theta + theta_dot * ts;
    double sn, cs;
    sincos(new_theta, &sn, &cs);
    s[0] = x + x_dot * ts; s[1] = x_dot + xacc * ts; s[2] = cs; s[3] = sn; s[4] = theta_dot + thetaacc * ts;
  } else {
    const double th1 = trig2angle(s[0], s[1]);
    const double th2 = trig2angle(s[2], s[3]);
    const double d1_ = s[4], d2_ = s[5];
    const double a0 = fmin(fmax(u[0], -5.0), 5.0), a1 = fmin(fmax(u[1], -5.0), 5.0);
    const double c2 = cos(th2), s2 = sin(th2);
    // m1 = m2 = l1 = I1 = I2 = 1, lc1 = lc2 = 0.5, g = 9.8 (oracle/dynamics.py)
    const double d1 = 0.25 + (1.0 + 0.25 + 1.0 * c2) + 1.0 + 1.0;
    const double d2 = (0.25 + 0.5 * c2) + 1.0;
    const double phi2 = 0.5 * 9.8 * cos(th1 + th2 - 1.5707963267948966);
    const double phi1 = -0.5 * (d2_ * d2_) * s2 - 1.0 * d2_ * d1_ * s2 + (0.5 + 1.0) * 9.8 * cos(th1 - 1.5707963267948966) + phi2;
    const double dd2 = (a0 + d2 / d1 * phi1 - 0.5 * (d1_ * d1_) * s2 - phi2) / (0.25 + 1.0 - d2 * d2 / d1);
    const double dd1 = -(a1 + d2 * dd2 + phi1) / d1;
    const double n1 = th1 + d1_ * ts, n2 = th2 + d2_ * ts;
    double sa, ca, sb, cb;
    sincos(n1, &sa, &ca);
    sincos(n2, &sb, &cb);
    s[0] = ca; s[1] = sa; s[2] = cb; s[3] = sb; s[4] = d1_ + dd1 * ts; s[5] = d2_ + dd2 * ts;
  }
}

}  // namespace nlc
