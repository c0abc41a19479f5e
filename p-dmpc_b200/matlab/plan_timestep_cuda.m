function infos = plan_timestep_cuda(handle, hlcs, mpa, options, time_step)
% PLAN_TIMESTEP_CUDA  All vehicles of one time step in ONE optimizer call on the GPU.
%
%   Replaces the level loop of PrioritizedSequentialController.controller
%   (hlc/controller/prioritized/PrioritizedSequentialController.m:74-92), in which every
%   vehicle's PrioritizedController.plan (PrioritizedController.m:297-352) runs one search after
%   reading the areas its sequential predecessors have published (consider_predecessors,
%   :449-506).  Here the searches of ALL vehicles are handed over at once; vehicle i waits ON
%   THE DEVICE for the vehicles j with directed_coupling_sequential(j, i) ~= 0 and takes their
%   planned areas as dynamic obstacles.  What an exhausted vehicle publishes depends only on the
%   previous time step (plan_fallback :678-718, handle_graph_search_exhaustion :568-621), so it
%   is passed up front as fallback_shapes.
%
%   handle : planner handle of pdmpc_b200_mex (GraphSearchCuda.handle)
%   hlcs   : 1 x N PrioritizedController objects, AFTER couple / prioritize / group of this time
%            step, i.e. hlcs(i).iter holds directed_coupling(_sequential)
%   infos  : 1 x N ControlResultsInfo, built by the reference's own helper
%            OptimizerInterface.create_control_results_info_from_mex (OptimizerInterface.m:63-101)
%
%   time_step : the time step PrioritizedController.plan passes to run_optimizer (:335-341); needed when
%            hlcs(1).optimizer is a MonteCarloTreeSearchCuda
%
%   Vehicles planning in PARALLEL to vehicle i (other groups) and its successors enter exactly as in
%   the reference: their reachable sets / previous trajectories / standstill areas are known
%   before the time step and are put into iter_v by the unchanged MATLAB code below.
%
%   With a MonteCarloTreeSearchCuda optimizer the searches are MonteCarloTreeSearch.run_optimizer's
%   (MEX command PLAN_TIMESTEP_SAMPLED): vehicle i's random stream has Seed = time_step + i
%   (MonteCarloTreeSearch.m:31), and its info is rebuilt as MonteCarloTreeSearchCuda.run_optimizer does.

    PLAN_TIMESTEP = 6;
    PLAN_TIMESTEP_SAMPLED = 13;
    N = numel(hlcs);
    Hp = options.Hp;
    x0 = zeros(N, 3); trims = zeros(N, 1); ref = zeros(N, Hp, 2); v_ref = zeros(N, Hp);
    obstacles = cell(N, 0); dyn = cell(N, 0, Hp); left = cell(N, 1); right = cell(N, 1);
    fallback_shapes = cell(N, Hp);
    coupling = hlcs(1).iter.directed_coupling_sequential;
    checker = double(~(options.scenario_type == ScenarioType.circle || ~options.is_prioritized));  % Config.m:71-87

    for i = 1:N
        c = hlcs(i);
        filter_self = false(1, options.amount); filter_self(i) = true;
        iter_v = IterationData.filter(c.iter, filter_self);                       % PrioritizedController.m:300-302
        predecessors = find(iter_v.directed_coupling(:, i) == 1)';
        sequential = find(iter_v.directed_coupling_sequential(:, i))';
        % parallel predecessors and successors: unchanged host logic (:391-447, :508-566)
        area_parallel = c.consider_predecessors(setdiff(predecessors, sequential), []);
        [obst_succ, area_succ] = c.consider_successors(find(iter_v.directed_coupling(i, :) == 1));
        obst_i = [iter_v.obstacles; obst_succ];
        % (+ the reachable sets of adjacent manual vehicles, InterX only: GraphSearchCuda.with_hdv_reachable_sets)
        iter_v.dynamic_obstacle_area = [iter_v.dynamic_obstacle_area; area_parallel; area_succ];
        dyn_i = GraphSearchCuda.with_hdv_reachable_sets(iter_v, checker, Hp);
        x0(i, :) = iter_v.x0(1, 1:3);
        trims(i) = iter_v.trim_indices;
        ref(i, :, :) = iter_v.reference_trajectory_points(1, :, :);
        v_ref(i, :) = iter_v.v_ref(1, :);
        obstacles(i, 1:numel(obst_i)) = obst_i(:)';
        dyn(i, 1:size(dyn_i, 1), :) = reshape(dyn_i, 1, size(dyn_i, 1), Hp);
        left{i} = iter_v.predicted_lanelet_boundary{1, 1};
        right{i} = iter_v.predicted_lanelet_boundary{1, 2};
        % what vehicle i publishes if its search is exhausted
        if mpa.trims(trims(i)).speed == 0 && options.constraint_from_successor ~= ConstraintFromSuccessor.none
            veh = c.scenario_adapter.scenario.vehicles(1);
            p = transformed_rectangle(x0(i, 1), x0(i, 2), x0(i, 3), veh.Length, veh.Width);   % :606-613
            fallback_shapes(i, :) = repmat({[p, p(:, 1)]}, 1, Hp);
        elseif ~isempty(c.info_old)
            fallback_shapes(i, :) = del_first_rpt_last(c.info_old.shapes);                  % :713
        end
    end

    args = {handle, x0, trims, ref, v_ref, obstacles, reshape(dyn, N, []), left, right, checker, options.dt_seconds, ...
        double(coupling), fallback_shapes};
    sampled = isa(hlcs(1).optimizer, 'MonteCarloTreeSearchCuda');
    if sampled
        [is_exhausted, n_expanded, trims_out, y, shapes, g, h] = pdmpc_b200_mex(PLAN_TIMESTEP_SAMPLED, args{:}, ...
            time_step + (1:N), hlcs(1).optimizer.n_expansions_max);
    else
        [is_exhausted, n_expanded, trims_out, y, shapes, g, h] = pdmpc_b200_mex(PLAN_TIMESTEP, args{:});
    end
    y = reshape(y, 3, Hp, N);

    infos = cell(1, N);
    for i = 1:N
        info = ControlResultsInfo(1, Hp);
        info.is_exhausted = logical(is_exhausted(i));
        info.n_expanded = n_expanded(i);
        if sampled && ~info.is_exhausted
            % path-only tree, as MonteCarloTreeSearchCuda.run_optimizer builds it (MonteCarloTreeSearch.m:207-239):
            % g = -1 except the goal leaf, h = -1
            tree = Tree();
            tree.trim = trims_out(i, :);
            tree.parent = uint32(0:Hp);
            tree.x = [x0(i, 1), y(1, :, i)];
            tree.y = [x0(i, 2), y(2, :, i)];
            tree.yaw = [x0(i, 3), y(3, :, i)];
            tree.k = 1:(Hp + 1);
            tree.g = [-1 * ones(1, Hp), g(i, end)];
            tree.h = -1 * ones(1, Hp + 1);
            info.tree = tree;
            info.tree_path = 1:(Hp + 1);
            info.y_predicted = y(:, :, i);
            info.shapes = shapes(i, :);
            info.predicted_trims = trims_out(i, 2:end);
            info.needs_fallback = false;
        elseif ~info.is_exhausted
            % next_nodes: Hp cells of 1 x 8 rows in NodeInfo order [x y yaw trim g h k exactEval]
            % (g, h: tree.get_cost(tree_path(end)) is what the explorative / optimal controllers compare,
            %  PrioritizedExplorativeController.m:100-104)
            next_nodes = arrayfun(@(k) [y(1, k, i), y(2, k, i), y(3, k, i), trims_out(i, k + 1), g(i, k + 1), h(i, k + 1), k, 1], ...
                1:Hp, UniformOutput = false);
            y_full = {[y(:, :, i)', trims_out(i, 2:end)']};
            iter_v = IterationData.filter(hlcs(i).iter, (1:options.amount) == i);
            info = OptimizerInterface.create_control_results_info_from_mex(info, iter_v, options, next_nodes, ...
                trims_out(i, :), y_full);
            info.shapes = shapes(i, :);
            info.needs_fallback = false;
        end
        infos{i} = info;   % exhausted vehicles: the caller runs handle_graph_search_exhaustion / plan_fallback as before
    end
end
