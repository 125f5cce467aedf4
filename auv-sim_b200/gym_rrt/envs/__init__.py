from gym_rrt.envs.rrt_env import DeviceVecRRTEnv, RRTEnv, VecRRTEnv  # noqa: F401
