"""Python mirror of the MPC seam: ocs2::SqpMpc as QMController::setupMpc builds it (qm_controllers/src/QMController.cpp:286-306):
one multiple-shooting SQP iteration per advanceMpc(), warm-started from the previous PrimalSolution."""
import numpy as np

from .interface import QMInterface, Solver


class SqpMpc:
    def __init__(self, interface=None, batch=1, device=0, time_horizon=0.0, dt=0.0, solver=None):
        self.solver = solver or Solver(interface or QMInterface(), batch=batch, device=device, time_horizon=time_horizon, dt=dt)
        self.batch = self.solver.batch

    def reset(self):
        """MPC_BASE::reset — forget the previous solution (cold start through QMInitializer)."""
        self.solver.mpc_reset()

    def run(self, prob):
        """MPC_BASE::run(t0, x0) for every robot; prob as in Solver.mpc_solve. Returns the PrimalSolution arrays."""
        return self.solver.mpc_solve(prob)

    def setFeedbackPolicy(self, on=True):
        """useFeedbackPolicy: the policy becomes the LinearController u = uff(t) + K(t) x of the last solve."""
        self.solver.mpc_set_feedback_policy(on)

    def evaluatePolicy(self, t, x=None):
        """MPC_MRT_Interface::evaluatePolicy(currentTime, currentState) → (optimizedState, optimizedInput, plannedMode).  Without a state the
        feed-forward policy is evaluated."""
        return self.solver.policy_eval(t) if x is None else self.solver.policy_eval_state(t, x)

    def setValueFunction(self, on=True):
        """createValueFunction: keep the value function of each solve's last QP."""
        self.solver.mpc_set_value_function(on)

    def getValueFunction(self, t, x):
        """SqpSolver::getValueFunction(time, state) of every robot → dict(f[B] = 0, dfdx[B, 30], dfdxx[B, 30, 30], valid[B]) (see Solver.value_function)."""
        v = self.solver.value_function(t, x); v["f"] = np.zeros(self.batch)
        return v

    def getLinearController(self, b0=0, count=None):
        """ocs2::LinearController of the last solve: dict(timeStamp[count, NMAX], biasArray, gainArray, feedback) (see Solver.mpc_get_controller)."""
        c = self.solver.mpc_get_controller(b0, count); sol = self.solver.mpc_get_solution(); n = len(c["feedback"])
        return dict(timeStamp=sol["t"][b0:b0 + n], n_nodes=sol["n_nodes"][b0:b0 + n], biasArray=c["bias"], gainArray=c["gain"], feedback=c["feedback"])
