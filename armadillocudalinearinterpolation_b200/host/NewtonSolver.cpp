// Newton iteration; behaviour follows NewtonSolver.cpp:40-245 of the reference: the parameter
// list is re-read at every Solve (so edits made after construction apply, Driver.cu:37), the
// residual history has maxIterations+1 slots, PostProcess() runs once after the loop, and the
// last Jacobian is copied out on request.  Two documented differences: the residual history IS
// trimmed to the iterations performed (the reference discards the result of head(), :134), and a
// singular Jacobian ends the solve as notConverged instead of throwing out of arma::solve.
#include "NewtonSolver.hpp"
#include <cassert>
#include <cmath>
#include <cstdlib>
#include <iostream>

NewtonSolver::NewtonSolver(AbstractNonlinearProblem* pProblem, const arma::vec* pInitialGuess,
                           const ParameterList* pParameterList)
    : mpProblem(pProblem), mpProblemJacobian(NULL), mpInitialGuess(pInitialGuess),
      mpParameterList(pParameterList), mpConvergenceCriterion(NULL), mMaxIterations(0),
      mPrintOutput(true), mTolerance(0.0), mFuse(true) {}

NewtonSolver::NewtonSolver(AbstractNonlinearProblem* pProblem,
                           AbstractNonlinearProblemJacobian* pProblemJacobian,
                           const arma::vec* pInitialGuess, const ParameterList* pParameterList)
    : mpProblem(pProblem), mpProblemJacobian(pProblemJacobian), mpInitialGuess(pInitialGuess),
      mpParameterList(pParameterList), mpConvergenceCriterion(NULL), mMaxIterations(0),
      mPrintOutput(true), mTolerance(0.0), mFuse(true) {}

NewtonSolver::~NewtonSolver() { delete mpConvergenceCriterion; }

void NewtonSolver::Initialise() {
  mMaxIterations = mpParameterList->maxIterations;
  mPrintOutput = mpParameterList->printOutput;
  mTolerance = mpParameterList->tolerance;
  if (mpConvergenceCriterion) mpConvergenceCriterion->SetTolerance(mTolerance);
  else mpConvergenceCriterion = new ConvergenceCriterion(mTolerance);
}

void NewtonSolver::Solve(arma::vec& solution, arma::vec& residualHistory, ExitFlagType& exitFlag,
                         arma::mat* pJacobianExternal) {
  Initialise();
  if (mPrintOutput) PrintHeader("Newton Method", mMaxIterations, mTolerance);

  const int n = (int)mpInitialGuess->n_rows;
  assert(n == (int)solution.n_rows);
  solution = *mpInitialGuess;

  // One object behind both interfaces that implements AbstractNonlinearProblemFused (EventDrivenMapB200): do not
  // evaluate F(u) twice per iteration.  Either the Jacobian is formed from the residual already in hand, or — when
  // the problem prefers it — F and dF/dU of every new iterate come in one batch (the Jacobian of an iterate that
  // turns out to be converged is then computed in vain).  `jacobian` stays the last Jacobian a step was taken with,
  // as in the reference (pJacobianExternal below).
  AbstractNonlinearProblemFused* fused = NULL;
  if (mFuse && mpProblemJacobian &&
      dynamic_cast<void*>(mpProblem) == dynamic_cast<void*>(mpProblemJacobian))
    fused = dynamic_cast<AbstractNonlinearProblemFused*>(mpProblemJacobian);
  const bool oneBatch = fused && fused->PrefersOneBatchPerIterate();

  arma::vec residual(n);
  arma::mat jacobian(n, n), jacobianAhead;
  if (oneBatch) { jacobianAhead.set_size(n, n); fused->ComputeFAndDFDU(solution, residual, jacobianAhead); }
  else mpProblem->ComputeF(solution, residual);
  double residualNorm = arma::norm(residual, 2);

  int iteration = 0;
  residualHistory.set_size(1 + mpParameterList->maxIterations);
  residualHistory(iteration) = residualNorm;
  if (mPrintOutput) PrintIteration(iteration, residualNorm, true);

  bool converged = mpConvergenceCriterion->TestConvergence(residualNorm);
  while (iteration < mMaxIterations && !converged) {
    if (oneBatch) jacobian = jacobianAhead;
    else if (fused) fused->ComputeDFDUGivenF(solution, residual, jacobian);
    else if (mpProblemJacobian) mpProblemJacobian->ComputeDFDU(solution, jacobian);
    else ComputeDFDU(solution, residual, jacobian);

    arma::vec direction;
    if (!arma::solve(direction, jacobian, -residual)) {
      if (mPrintOutput) std::cout << "Newton: singular Jacobian, stopping" << std::endl;
      break;
    }
    solution += mpParameterList->damping * direction;
    iteration++;

    if (oneBatch) fused->ComputeFAndDFDU(solution, residual, jacobianAhead);
    else mpProblem->ComputeF(solution, residual);
    residualNorm = arma::norm(residual, 2);
    converged = mpConvergenceCriterion->TestConvergence(residualNorm);
    residualHistory(iteration) = residualNorm;
    if (mPrintOutput) PrintIteration(iteration, residualNorm);
  }

  PostProcess();
  residualHistory = residualHistory.head(iteration + 1);
  exitFlag = converged ? ExitFlagType::converged : ExitFlagType::notConverged;
  if (mPrintOutput) PrintFooter(iteration, exitFlag);

  if (pJacobianExternal) {
    assert((int)pJacobianExternal->n_rows == n && (int)pJacobianExternal->n_cols == n);
    *pJacobianExternal = jacobian;
  }
}

// Forward differences, one ComputeF per column: J(:, i) = (F(u + eps e_i) - F(u)) * eps^-1
void NewtonSolver::ComputeDFDU(const arma::vec& u, const arma::vec& f, arma::mat& jacobian) {
  const int n = (int)mpInitialGuess->n_rows;
  const double epsilon = mpParameterList->finiteDifferenceEpsilon;
  arma::vec perturbed(u);
  arma::vec fPerturbed(n);
  for (int i = 0; i < n; i++) {
    if (i > 0) perturbed(i - 1) = u(i - 1);
    perturbed(i) += epsilon;
    mpProblem->ComputeF(perturbed, fPerturbed);
    jacobian.col(i) = (fPerturbed - f) * std::pow(epsilon, -1);
  }
}

void NewtonSolver::SetInitialGuess(const arma::vec* pInitialGuess) { mpInitialGuess = pInitialGuess; }
void NewtonSolver::SetParameterList(const ParameterList* pParameterList) { mpParameterList = pParameterList; }
void NewtonSolver::SetProblem(AbstractNonlinearProblem* pProblem) { mpProblem = pProblem; }
void NewtonSolver::SetProblemJacobian(AbstractNonlinearProblemJacobian* pProblemJacobian) {
  mpProblemJacobian = pProblemJacobian;
}
void NewtonSolver::PostProcess() { mpProblem->PostProcess(); }
