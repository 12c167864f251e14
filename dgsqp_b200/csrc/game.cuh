// Selects the game the solver stack is compiled for.  The solver (qp_gi.cuh, lsqr.cuh, sqp_v1.cuh, sqp_v2.cuh) sees a
// game only through: GameDesc, Dims/make_dims, EvalBuf, DG_AB_SZ / DG_T2_SZ / DG_HC_SZ (per-(stage, agent) sizes of
// the derivative tables), game_bind, game_row_table, game_rollout, game_linearize, game_constraints, game_costates,
// game_sens, game_contract, game_gradients, game_hessian, game_G_times, game_GT_times, game_G_row, game_G_cols,
// game_G_sparse, game_costs.
// One translation unit = one game (dgsqp_abi.cu: racing games; dgsqp_merge_abi.cu: merge game, -DDG_GAME_MERGE).
//
// Most of that interface is written once: game_layout.cuh (row layout, EvalTables, sensitivity packing) and
// game_kkt.cuh (constraints, G products, costates, gradients, Hessian DP).  A game header provides
//   - DG_NQA, DG_NUA, DG_T2_SZ, DG_HC_SZ, DG_GAME_ROWS, DG_GAME_ROWS_N, DG_BOUND_STATE and GameDesc, then includes
//     game_layout.cuh and defines EvalBuf (deriving from EvalTables) and game_bind;
//   - game_rollout, game_linearize, game_costs and the contraction look-ups hc_xx / hc_ux / hc_uu;
//   - the forceinline hooks that game_kkt.cuh calls, then includes game_kkt.cuh:
//       game-specific rows (K_GAME):  RowCoef, game_row_value, game_row_Gv, game_row_prep + game_row_G (one entry of
//         G), game_row_sparse (its +-1 entries, if any), game_row_coefs (its part of the state coefficients of G' w),
//         game_row_GT_direct (its part of G' w on the inputs), game_row_lx (its part of d(l'C)/dx);
//       state-bound values:  game_state_ub, game_state_lb;
//       costs:  game_term_lx / game_stage_lx and game_term_lxx / game_stage_lxx (state cost gradient and Hessian of
//         agent f at k = N and at 1 <= k < N), InputGrad + game_input_grad + input_grad_plus (input-cost gradient,
//         added to the two sums of game_gradients), game_input_hess, game_input_hess_prev (the Hessian entry between
//         u_k and u_{k-1} of the same agent and input), game_contract_entry (one entry of p' T2).
// A hook whose game has no such term returns a literal 0.0 (or false, or does nothing), so the compiler removes it.
#pragma once
#ifdef DG_GAME_MERGE
#include "merge_game.cuh"
#else
#include "racing_game.cuh"
#endif
