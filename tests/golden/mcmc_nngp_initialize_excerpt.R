# The lines of the reference's Scripts/mcmc_nngp_initialize.R that R/patches/mcmc_nngp_initialize.patch changes: each hunk's
# context and removed lines, verbatim, in file order (reference lines 90-96, 107-113 and 198-211).  Stored so that the patch can
# be checked against them without the reference tree (tests/test_r_glue_cpu.py).
    # count how many observations correspond to one location
    vecchia_approx$obs_per_loc = unlist(sapply(vecchia_approx$hctam_scol, length))
    #extracting NNarray =  nearest neighbours for Vecchia approximation
    vecchia_approx$NNarray = GpGp::find_ordered_nn(locs, m)
    
    #computations from vecchia_approx$NNarray in order to create sparse Cholesky using Matrix::sparseMatrix
    #non_NA indices from vecchia_approx$NNarray
    vecchia_approx$MRF_adjacency_mat[1, 2] = 0
    vecchia_approx$MRF_adjacency_mat[1, 2] = 1
    vecchia_approx$MRF_adjacency_mat@x = rep(1, length(vecchia_approx$MRF_adjacency_mat@x))
    vecchia_approx$coloring = naive_greedy_coloring(vecchia_approx$MRF_adjacency_mat)
    
    ##############
    # Regressors #
          if(substr(space_time_model$covfun$shape_params[j], 1, 3)=="log")return(exp(states[[i]]$params$shape[j]))
          else if(substr(space_time_model$covfun$shape_params[j], 1, 6)=="qlogis")return(.4+.7*plogis(states[[i]]$params$shape[j]))
        })
        Linv = GpGp::vecchia_Linv(covparms = c(1, shape, 0), covfun_name = stationary_covfun, locs = locs, NNarray = vecchia_approx$NNarray)
        Linv = 
          Matrix::sparseMatrix(
            i = vecchia_approx$sparse_chol_row_idx, 
            j = vecchia_approx$sparse_chol_column_idx, 
            x = Linv[vecchia_approx$NNarray_non_NA], 
            triangular = T)
        states[[i]]$params$field  = states[[i]]$params$beta_0 + sqrt(exp(states[[i]]$params$log_scale)) * as.vector(Matrix::solve(Linv, rnorm(vecchia_approx$n_locs)))
      }
    }

