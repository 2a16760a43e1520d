// oracle/ros_ref_driver.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// C entry points into the reference's UNMODIFIED ROS-side sources (mpc_ros/src/driving_state.cpp,
// mpc_ros/src/mpc_planner_ros.cpp), compiled from /root/reference against the stand-in ROS / Eigen headers in
// shim/ros_stubs and shim/Eigen and linked with the reference's own mpc_planner.cpp (oracle/_ref):
//   * ros_ref_window      : MPCPlannerROS::getCutOffPlan (:266-291) + downSamplePlan (:365-391)
//   * ros_ref_tick_*      : DrivingStateContext + Tracking::mpcComputeVelocityCommands (driving_state.cpp:105-119):
//                           deceleration (:121-141), findBestPath (:175-271) incl. transform, polyfit, state assembly,
//                           MPC::Solve, speed clamp
// With them, oracle/mpc_oracle.c's restatement of those functions can be compared with the reference's own code.
// (the standard / stub headers first, so that only the reference's own classes are opened up)
#include <cmath>
#include <cstring>
#include <fstream>
#include <iostream>
#include <map>
#include <sstream>
#include <string>
#include <vector>
#include <Eigen/Dense>
#include "ros/ros.h"
#include <nav_core/base_local_planner.h>
#include <base_local_planner/trajectory.h>
#include <base_local_planner/local_planner_util.h>
#include <base_local_planner/goal_functions.h>
#include <costmap_2d/costmap_2d_ros.h>
#include <dynamic_reconfigure/server.h>
#include <mpc_ros/MPCPlannerConfig.h>
#include <angles/angles.h>
#include <tf2_geometry_msgs/tf2_geometry_msgs.h>
#include <tf2_ros/buffer.h>
#include <nav_msgs/Odometry.h>
#include <std_msgs/String.h>
#include "mpc_planner.h"
#define private public      // the windowing helpers are private members of MPCPlannerROS
#define protected public
#include "mpc_planner_ros.h"
#undef private
#undef protected

#include <cmath>
#include <cstring>

static geometry_msgs::PoseStamped make_pose(double x, double y, double yaw)
{
    geometry_msgs::PoseStamped p;
    p.pose.position.x = x; p.pose.position.y = y;
    p.pose.orientation.z = std::sin(0.5 * yaw); p.pose.orientation.w = std::cos(0.5 * yaw);
    return p;
}

extern "C" {

// Returns the number of down-sampled waypoints written to out_x / out_y (capacity cap), or -1 when the reference
// reports failure; *n_erased = plan points getCutOffPlan removed from the front.  path_length is what the reference's
// uninitialised _pathLength would have to hold; _waypointsDist starts at -1 (the cfg default, MPCPlanner.cfg:18), so
// the spacing is measured from the plan as downSamplePlan does (:369-375).
int ros_ref_window(int n, const double *px, const double *py, double rx, double ry, double path_length, int cap,
                   double *out_x, double *out_y, int *n_erased, int *down_sampling)
{
    static mpc_ros::MPCPlannerROS *planner = new mpc_ros::MPCPlannerROS();
    std::vector<geometry_msgs::PoseStamped> plan;
    for (int i = 0; i < n; i++) plan.push_back(make_pose(px[i], py[i], 0.0));
    const geometry_msgs::PoseStamped robot = make_pose(rx, ry, 0.0);
    const bool ok = planner->getCutOffPlan(robot, plan);
    if (n_erased) *n_erased = n - (int)plan.size();
    if (!ok || plan.size() < 2) return -1;
    planner->_pathLength = path_length;
    planner->_waypointsDist = -1.0;
    planner->_downSampling = 0;
    std::vector<geometry_msgs::PoseStamped> ds;
    planner->downSamplePlan(ds, plan);
    if (down_sampling) *down_sampling = planner->_downSampling;
    int m = 0;
    for (size_t i = 0; i < ds.size() && m < cap; i++, m++) { out_x[m] = ds[i].pose.position.x; out_y[m] = ds[i].pose.position.y; }
    return (int)ds.size();
}

struct RosRefTracker {
    DrivingStateContext *ctx;
    Tracking *tracking;
};

// cfg: the 15 LoadParams values in the key order of driving_state.cpp:65-79 (DT first) -- DT, STEPS, REF_CTE, REF_ETHETA,
// REF_V, W_CTE, W_EPSI, W_V, W_ANGVEL, W_A, W_DANGVEL, W_DA, ANGVEL, MAXTHR, BOUND.
void *ros_ref_tick_new(const double *cfg15, int delay_mode, double max_speed)
{
    // the reference announces itself on std::cout ("init mpc", the context's parameter dump): kept off the harness output
    std::streambuf *old = std::cout.rdbuf();
    std::ostringstream sink;
    std::cout.rdbuf(sink.rdbuf());
    RosRefTracker *t = new RosRefTracker();
    t->ctx = new DrivingStateContext();
    t->tracking = new Tracking(t->ctx);
    t->ctx->transitionTo(t->tracking);
    t->ctx->updateControlFrequency(cfg15[0]);
    mpc_ros::MPCPlannerConfig c;
    c.debug_info = false; c.delay_mode = delay_mode != 0;
    c.steps = cfg15[1]; c.ref_cte = cfg15[2]; c.ref_etheta = cfg15[3]; c.ref_vel = cfg15[4];
    c.w_cte = cfg15[5]; c.w_etheta = cfg15[6]; c.w_vel = cfg15[7]; c.w_angvel = cfg15[8]; c.w_accel = cfg15[9];
    c.w_angvel_d = cfg15[10]; c.w_accel_d = cfg15[11]; c.max_angvel = cfg15[12]; c.max_throttle = cfg15[13];
    c.bound_value = cfg15[14];
    t->ctx->updateMpcConfigs(c);
    t->ctx->_max_speed = max_speed;
    std::cout.rdbuf(old);
    return t;
}

// previous w / throttle (delay compensation, driving_state.cpp:191-192) and REF_V persist in the context between ticks;
// state_io = {_w, _throttle, REF_V} lets the caller set them before and read them after the tick.
// out5 = {cmd linear.x, cmd angular.z, _w, _throttle, REF_V}; pred (3 x N, may be NULL) = mpc_x, mpc_y, mpc_theta.
int ros_ref_tick(void *h, double px, double py, double yaw, double gx, double gy, double v_feedback,
                 int m, const double *wx, const double *wy, double *state_io3, double *out5, double *pred, int npred)
{
    RosRefTracker *t = (RosRefTracker *)h;
    if (state_io3) {
        t->ctx->_w = state_io3[0]; t->ctx->_throttle = state_io3[1];
        t->ctx->mpc_params_["REF_V"] = state_io3[2];
        t->ctx->_mpc.LoadParams(t->ctx->mpc_params_);
    }
    std::vector<geometry_msgs::PoseStamped> plan;
    for (int i = 0; i < m; i++) plan.push_back(make_pose(wx[i], wy[i], 0.0));
    geometry_msgs::Twist fb; fb.linear.x = v_feedback;
    geometry_msgs::Twist cmd;
    const bool ok = t->ctx->getCmd(cmd, make_pose(px, py, yaw), make_pose(gx, gy, 0.0), fb, plan);
    out5[0] = cmd.linear.x; out5[1] = cmd.angular.z; out5[2] = t->ctx->_w; out5[3] = t->ctx->_throttle;
    out5[4] = t->ctx->mpc_params_["REF_V"];
    if (state_io3) { state_io3[0] = t->ctx->_w; state_io3[1] = t->ctx->_throttle; state_io3[2] = out5[4]; }
    if (pred) {
        const std::vector<double> &x = t->ctx->_mpc.mpc_x, &y = t->ctx->_mpc.mpc_y, &th = t->ctx->_mpc.mpc_theta;
        for (int k = 0; k < npred; k++) {
            pred[k] = k < (int)x.size() ? x[k] : 0.0;
            pred[npred + k] = k < (int)y.size() ? y[k] : 0.0;
            pred[2 * npred + k] = k < (int)th.size() ? th[k] : 0.0;
        }
    }
    return ok ? 1 : 0;
}

// the reference's free functions (driving_state.cpp:273-300)
void ros_ref_polyfit(int m, const double *x, const double *y, int order, double *coeffs_out)
{
    Eigen::VectorXd xv(m), yv(m);
    for (int i = 0; i < m; i++) { xv[i] = x[i]; yv[i] = y[i]; }
    Eigen::VectorXd c = polyfit(xv, yv, order);
    for (int i = 0; i <= order; i++) coeffs_out[i] = c[i];
}

double ros_ref_polyeval(int nc, const double *coeffs, double x)
{
    Eigen::VectorXd c(nc);
    for (int i = 0; i < nc; i++) c[i] = coeffs[i];
    return polyeval(c, x);
}

}  // extern "C"
